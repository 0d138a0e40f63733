// api.cu — host orchestration and the C ABI (include/xpng_b200.h) of the B200 xPNG codec.
// Everything here is plumbing: tile tables (libxpng.c:51-83), scratch layout, kernel launches, host<->device
// copies.  All codec arithmetic lives in the kernels.
//
// Execution model.  A context owns LANES: a lane is a set of CUDA streams plus its own scratch buffers.  A call
// cuts its batch into chunks of whole images and issues every chunk on its own lane WITHOUT waiting for it; only at
// the end does the host collect the per-chunk size tables (encode) or error flags (decode).  The serial chains of the
// bit stream (rANS recurrences, context walk) leave most of the machine idle while they run; with several chunks
// in flight the data-parallel kernels of one chunk fill the SMs under the chains of another, and with host buffers the
// H2D / D2H copies of one chunk overlap the kernels of its neighbours.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <vector>

#include "../../include/xpng_b200.h"
#include "common.cuh"
#include "enc_front.cuh"
#include "enc_front2.cuh"
#include "enc_back.cuh"
#include "enc_m2.cuh"
#include "enc_rans_lat.cuh"
#include "enc_order.cuh"
#include "dec_m1.cuh"
#include "dec_back.cuh"
#include "dec_rans_lat.cuh"
#include "dec_rans_pair.cuh"
#include "dec_walk3.cuh"
#include "misc.cuh"
#include "orient.cuh"
#include "region.cuh"
#include "resize.cuh"
#include "tensor.cuh"
#include "color.cuh"
#include "blur.cuh"
#include "augment.cuh"

using namespace xpb;

struct DevBuf { void* p = nullptr; size_t cap = 0; };
struct PinBuf { void* p = nullptr; size_t cap = 0; };

struct xpngb_ctx {
    int device = 0;
    xpngb_ctx* root = nullptr;                 // the context the caller holds: error text, launch counter, profile table, tunables
    std::vector<xpngb_ctx*> lanes;             // root only: further lanes (lane 0 is the root itself), created on demand
    static constexpr int NSIDE = 5;
    cudaStream_t stream = nullptr, side[NSIDE] = {}, cur = nullptr;   // main stream, side streams for independent chains, stream of the next launch
    cudaStream_t hi = nullptr;                 // high-priority twin of the main stream: serial-chain kernels (LAUNCH_HI)
    cudaEvent_t ev_hi = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join[NSIDE] = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, pe0 = nullptr, pe1 = nullptr, ev_done = nullptr;
    int profile = 0;   // 1: per-kernel CUDA-event timing accumulated (serialises the launches); 2: also print to stderr;
                       // 3: timeline — start/end of every launch relative to the call's start, launches NOT serialised (stderr)
    int lane_id = 0;
    struct TlRow { const char* name; int lane; cudaEvent_t a, b; };
    std::vector<TlRow> tl;
    struct ProfRow { const char* name; double ms; uint32_t count; };
    std::vector<ProfRow> prof;
    char err[512] = { 0 };
    float last_ms = 0.f;
    uint32_t launches = 0;
    uint64_t decoded_tiles = 0;               // tiles the last decode call decoded, over all its chunks (xpngb_last_tiles)
    uint64_t max_chunk_px = 1ull << 30;       // XPNGB_CHUNK_MPIX: upper bound of a chunk (bounds the scratch of a lane)
    uint32_t pipe_lanes = 8;                  // XPNGB_PIPE_LANES: chunks in flight per call
    uint64_t pipe_min_px = 32ull << 20;       // XPNGB_PIPE_MIN_MPIX: no chunk smaller than this
    bool walk_ring = false;                   // XPNGB_WALK=ring: force the ring walk (tests)
    uint32_t direct_max_tiles = 148;  // level-2 decode: tiles per call up to which the 64 KiB direct tables are used (3 chains per SM stay resident)
    uint32_t v2_direct_max_tiles = ~0u;  // level-1 decode: same trade for the 16 KiB context tables
    uint32_t unr_multi_max_tiles = 592;  // un-predict: tiles per call up to which a tile gets 8 warps
    uint32_t s16_lat_max_tiles = 1776;  // level-2 decode, pair family: calls up to this many tiles decode the 16-symbol value stream (the longest chain) warp-per-block
    uint32_t lat_max_blocks = 12000;  // decode: entropy blocks per call up to which the warp-per-block (latency) kernels are used (measured crossover, profiles/)
    // device scratch
    DevBuf pixels, norm, files, arena, tiles, imgs, seg_tile, costs, hist, seginfo, place, vplace, vcnt, sym_area,
        bits_area, alpha, streams, blocks, state, outs, flags, skip, dimgs, dtiles, plane, nlseq, rowcnt, rowbits, eord,
        rows, edge, errflag, hdr, offs, m2a, m2b, tclass, tabs, ccnt, cbit, resv, oriented, odesc, pdw,
        region, crops,   // region decode: window of the selected tiles, crop descriptors
        orients,         // oriented decode: OrientDesc of the lane's chunk (odesc belongs to xpngb_transform / encode_oriented)
        rdescs, rtab, rtmp,   // resized decode: ResizeDesc of the lane's chunk, windows and weights, the first pass's rows
        tdescs, tsrc,         // tensor decode: TensorDesc of the lane's chunk, the resized (and coloured) entries' pixels
        cdescs,               // colour decode: ColorDesc of the lane's chunk, then one 64-bit luma sum per descriptor
        bdescs, bscr,         // blurred decode: BlurPass of the lane's chunk, the second buffer of each entry's ping-pong
        adescs;               // augmented decode: the chunk's AugPix, ColorDesc, luma sums, AugLut and histograms, stage by stage
    PinBuf pin_a, pin_b, pin_o;   // pin_o: orientation descriptors (their upload may still be in flight when an encode reuses pin_a)
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            snprintf(ctx->root->err, sizeof ctx->root->err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)
#define FAIL(...)                                                            \
    do {                                                                     \
        snprintf(ctx->root->err, sizeof ctx->root->err, __VA_ARGS__);        \
        return 1;                                                            \
    } while (0)
#define LAUNCH(kernel, grid, block, smem, ...)                                                      \
    do {                                                                                            \
        xpngb_ctx* r_ = ctx->root;                                                                  \
        if (r_->profile == 3) tl_mark(ctx, #kernel, 0);                                             \
        else if (r_->profile) cudaEventRecord(ctx->pe0, ctx->cur);                                  \
        kernel<<<grid, block, smem, ctx->cur>>>(__VA_ARGS__);                                       \
        r_->launches++;                                                                             \
        CK(cudaGetLastError());                                                                     \
        if (r_->profile == 3) tl_mark(ctx, #kernel, 1);                                             \
        else if (r_->profile) {                                                                          \
            float ms_ = 0; cudaEventRecord(ctx->pe1, ctx->cur); cudaEventSynchronize(ctx->pe1);     \
            cudaEventElapsedTime(&ms_, ctx->pe0, ctx->pe1);                                         \
            prof_add(r_, #kernel, ms_);                                                             \
            if (r_->profile > 1) fprintf(stderr, "[xpngb] %-28s %9.3f ms\n", #kernel, ms_);       \
        }                                                                                           \
    } while (0)

// Independent serial chains (e.g. the value-stream blocks of level 2 while the context streams are walked)
// run on the side stream: FORK makes it wait for everything launched so far, JOIN makes the main stream wait for it.
// Chain kernels (rANS recurrences, context walks, the tiny serial scans between them) keep a few warps busy for a long
// time; the data-parallel kernels of the other chunks in flight fill the machine.  The block scheduler serves streams
// of higher priority first, so chains go to high-priority streams: their CTAs become resident as soon as they are
// launched instead of queueing behind hundreds of thousands of front-end CTAs.
// level 0: the longest chains of a call (side stream 0: the 16-symbol value streams of level 2), level 1: other chains.
static cudaStream_t prio_stream(const xpngb_ctx* ctx, int level) {
    cudaStream_t s = nullptr;
    int lo = 0, hi = 0;   // numerically lower = served first
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess && hi != lo)
        cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, (hi + level < lo) ? hi + level : hi);
    else cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    return s;
}
static cudaStream_t side_of(xpngb_ctx* ctx, int k) {
    if (!ctx->side[k]) ctx->side[k] = prio_stream(ctx, k == 0 ? 0 : 1);   // side streams only ever carry chains
    return ctx->side[k];
}
#define LAUNCH_HI(kernel, grid, block, smem, ...)                                                   \
    do {                                                                                            \
        cudaStream_t base_ = ctx->cur;                                                              \
        const bool tw_ = base_ == ctx->stream && (ctx->root->profile == 0 || ctx->root->profile == 3);       \
        if (tw_) {                                                                                  \
            if (!ctx->hi) ctx->hi = prio_stream(ctx, 1);                                               \
            CK(cudaEventRecord(ctx->ev_hi, base_)); CK(cudaStreamWaitEvent(ctx->hi, ctx->ev_hi, 0)); ctx->cur = ctx->hi; \
        }                                                                                           \
        LAUNCH(kernel, grid, block, smem, __VA_ARGS__);                                             \
        if (tw_) { CK(cudaEventRecord(ctx->ev_hi, ctx->hi)); CK(cudaStreamWaitEvent(base_, ctx->ev_hi, 0)); ctx->cur = base_; } \
    } while (0)
#define FORK_SIDE(k) FORK_FROM(ctx->stream, k)
#define FORK_FROM(src, k) do { CK(cudaEventRecord(ctx->ev_fork, (src))); CK(cudaStreamWaitEvent(side_of(ctx, k), ctx->ev_fork, 0)); ctx->cur = ctx->side[k]; } while (0)
#define BACK_TO_MAIN() do { ctx->cur = ctx->stream; } while (0)
#define JOIN_SIDE(k) do { ctx->cur = ctx->stream; CK(cudaEventRecord(ctx->ev_join[k], ctx->side[k])); CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[k], 0)); } while (0)

// Timeline mode: two events around a launch on its own stream (no host wait); tl_dump prints them after the call.
static void tl_mark(xpngb_ctx* ctx, const char* name, int end) {
    xpngb_ctx* r = ctx->root;
    if (!end) {
        xpngb_ctx::TlRow row{ name, ctx->lane_id, nullptr, nullptr };
        cudaEventCreate(&row.a); cudaEventCreate(&row.b);
        cudaEventRecord(row.a, ctx->cur);
        r->tl.push_back(row);
    } else cudaEventRecord(r->tl.back().b, ctx->cur);
}
static void tl_dump(xpngb_ctx* ctx, const char* what) {
    if (ctx->profile != 3) return;
    cudaDeviceSynchronize();
    for (auto& row : ctx->tl) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, ctx->ev0, row.a); cudaEventElapsedTime(&b, ctx->ev0, row.b);
        fprintf(stderr, "TL %s %d %s %.3f %.3f\n", what, row.lane, row.name, a, b);
        cudaEventDestroy(row.a); cudaEventDestroy(row.b);
    }
    ctx->tl.clear();
}
static void prof_add(xpngb_ctx* ctx, const char* name, float ms) {
    for (auto& r : ctx->prof) if (!strcmp(r.name, name)) { r.ms += ms; r.count++; return; }
    ctx->prof.push_back({ name, ms, 1 });
}

static int ensure(xpngb_ctx* ctx, DevBuf& b, size_t n) {
    n += 64;   // tail slack for vector over-reads
    if (b.cap >= n) return 0;
    if (b.p) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = n + n / 8;
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    return 0;
}
static int ensure_pin(xpngb_ctx* ctx, PinBuf& b, size_t n) {
    if (b.cap >= n) return 0;
    if (b.p) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFreeHost(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = n + n / 8 + 4096;
    CK(cudaMallocHost(&b.p, want));
    b.cap = want;
    return 0;
}
#define ENSURE(buf, n) do { if (ensure(ctx, ctx->buf, (n))) return 1; } while (0)

// ------------------------------------------------------------------------------------------------
// Tile grid (libxpng.c:51-83): base tile 444x444 (or full width/height when the image is thinner),
// the remainder of each axis goes to the first tile, or to the first two when it exceeds half a tile.
// The grid is part of the format: the encoder, the decoder and region selection all take it from tile_grid.
// ------------------------------------------------------------------------------------------------
static uint64_t axis_cut(uint64_t extent, uint64_t base, uint64_t* first, uint64_t* second) {
    uint64_t n = extent / base, rem = extent % base;
    *first = base + rem; *second = base;
    if (rem > base / 2) { n++; *second = (base + rem) / 2; *first = *second + ((base + rem) & 1); }
    return n;
}

struct TileGrid {
    uint64_t nw = 1, nh = 1, w0, w1, wb, h0, h1, hb;   // tiles per row / column; sizes of the first, second and other tiles
    // start / size of tile k along an axis whose first two tiles are a and b long and the others base long
    static uint64_t start(uint64_t k, uint64_t a, uint64_t b, uint64_t base) { return k == 0 ? 0 : (k == 1 ? a : a + b + (k - 2) * base); }
    static uint64_t size(uint64_t k, uint64_t a, uint64_t b, uint64_t base) { return k == 0 ? a : (k == 1 ? b : base); }
    static uint64_t at(uint64_t v, uint64_t n, uint64_t a, uint64_t b, uint64_t base) {   // the tile that holds pixel v
        const uint64_t k = v < a ? 0 : (v - a < b ? 1 : 2 + (v - a - b) / base);
        return k < n ? k : n - 1;
    }
    uint64_t x_of(uint64_t j) const { return start(j, w0, w1, wb); }
    uint64_t y_of(uint64_t i) const { return start(i, h0, h1, hb); }
    uint64_t w_of(uint64_t j) const { return size(j, w0, w1, wb); }
    uint64_t h_of(uint64_t i) const { return size(i, h0, h1, hb); }
    uint64_t col_at(uint64_t x) const { return at(x, nw, w0, w1, wb); }
    uint64_t row_at(uint64_t y) const { return at(y, nh, h0, h1, hb); }
};

static TileGrid tile_grid(uint64_t W, uint64_t H) {
    TileGrid g;
    g.w0 = g.w1 = g.wb = W; g.h0 = g.h1 = g.hb = H;
    if (W * H > TILE_AREA) {
        if (W < 444) { g.wb = W; g.hb = TILE_AREA / W; }
        else if (H < 444) { g.hb = H; g.wb = TILE_AREA / H; }
        else g.wb = g.hb = 444;
        g.nw = axis_cut(W, g.wb, &g.w0, &g.w1);
        g.nh = axis_cut(H, g.hb, &g.h0, &g.h1);
    }
    return g;
}

struct TileSel { uint64_t r0, r1, c0, c1; };   // tile rows [r0, r1] and tile columns [c0, c1] of a grid
static TileSel all_tiles(const TileGrid& g) { return TileSel{ 0, g.nh - 1, 0, g.nw - 1 }; }

// The tiles a region decode of r (inside a W x H image) decodes, and their union `cover` (whole tiles, image pixels).
// False when r is empty or not inside the image; x + w > W is tested without overflow.
static bool region_select(uint64_t W, uint64_t H, const xpngb_rect& r, TileGrid& g, TileSel& s, xpngb_rect& cover) {
    if (!W || !H || W > (1u << 24) || H > (1u << 24)) return false;
    if (!r.w || !r.h || r.x >= W || r.w > W - r.x || r.y >= H || r.h > H - r.y) return false;
    g = tile_grid(W, H);
    s = TileSel{ g.row_at(r.y), g.row_at(r.y + r.h - 1), g.col_at(r.x), g.col_at(r.x + r.w - 1) };
    cover.x = g.x_of(s.c0); cover.y = g.y_of(s.r0);
    cover.w = g.x_of(s.c1) + g.w_of(s.c1) - cover.x; cover.h = g.y_of(s.r1) + g.h_of(s.r1) - cover.y;
    return true;
}

extern "C" uint32_t xpngb_region_tiles(uint64_t w, uint64_t h, const xpngb_rect* r, xpngb_rect* cover) {
    TileGrid g; TileSel s; xpngb_rect c{};
    if (!r || !region_select(w, h, *r, g, s, c)) return 0;
    if (cover) *cover = c;
    return (uint32_t)((s.r1 - s.r0 + 1) * (s.c1 - s.c0 + 1));
}

struct Plan {
    std::vector<ImageDesc> imgs;
    std::vector<TileDesc> tiles;
    std::vector<uint32_t> seg_tile;
    uint64_t px_total = 0, row_total = 0, str_total = 0, blk_total = 0;
    bool any_rgba = false;
    bool any_wide = false;     // a tile wider than the staged front end takes (one-tile images up to 197136 x 1)
};

// Appends the selected tiles of one W x H image.  Tile (x0, y0) is read (encode) or written (decode) at
// D + (y0 - oy) * Pd + (x0 - ox) * pxsz: the image itself (D = its pixels, Pd = W * pxsz, origin 0), or for a region
// decode a window of row pitch Pd whose first pixel is image pixel (ox, oy).
static void plan_image(Plan& P, const TileGrid& g, const TileSel& s, uint64_t D, uint64_t Pd, uint64_t ox, uint64_t oy,
                       uint64_t W, uint64_t H, uint32_t pxsz, uint32_t mode, int sfac, int bfac) {
    ImageDesc I{};
    I.px_off = D; I.raw_size = W * H * pxsz; I.w = (uint32_t)W; I.h = (uint32_t)H; I.pxsz = pxsz;
    I.tile0 = (uint32_t)P.tiles.size(); I.mode = mode;
    const uint32_t img = (uint32_t)P.imgs.size();
    uint64_t y = g.y_of(s.r0);
    for (uint64_t i = s.r0; i <= s.r1; i++) {
        const uint64_t th = g.h_of(i);
        uint64_t x = g.x_of(s.c0);
        for (uint64_t j = s.c0; j <= s.c1; j++) {
            const uint64_t tw = g.w_of(j);
            TileDesc t{};
            t.src_off = D + (y - oy) * Pd + (x - ox) * pxsz;
            t.px_off = P.px_total; t.row_off = P.row_total;
            t.w = (uint32_t)tw; t.h = (uint32_t)th; t.bpr = (uint32_t)Pd; t.npx = (uint32_t)(tw * th);
            t.img = img; t.seg0 = (uint32_t)P.seg_tile.size(); t.nseg = (t.npx + SEG - 1) / SEG; t.pxsz = pxsz;
            t.x0 = (uint32_t)x; t.y0 = (uint32_t)y; t.tix = (uint32_t)(i * g.nw + j);
            const uint64_t slice = ((uint64_t)t.npx + 15) / 16 * 16 + 256;
            t.str_off = P.str_total; t.blk_off = P.blk_total;
            P.px_total += slice; P.row_total += th;
            P.str_total += slice * sfac; P.blk_total += slice * bfac + 8192;
            for (uint32_t k = 0; k < t.nseg; k++) P.seg_tile.push_back((uint32_t)P.tiles.size());
            if (t.w > FRONT2_MAXW) P.any_wide = true;
            P.tiles.push_back(t);
            x += tw;
        }
        y += th;
    }
    I.ntiles = (uint32_t)P.tiles.size() - I.tile0;
    if (pxsz == 4) P.any_rgba = true;
    P.imgs.push_back(I);
}

// Every tile of an image, in place.  base = absolute device address of its pixels.
static void plan_image(Plan& P, uint64_t base, uint64_t W, uint64_t H, uint32_t pxsz, uint32_t mode, int sfac, int bfac) {
    const TileGrid g = tile_grid(W, H);
    plan_image(P, g, all_tiles(g), base, W * pxsz, 0, 0, W, H, pxsz, mode, sfac, bfac);
}

static int upload_plan(xpngb_ctx* ctx, const Plan& P) {
    const size_t nb_t = P.tiles.size() * sizeof(TileDesc), nb_i = P.imgs.size() * sizeof(ImageDesc), nb_s = P.seg_tile.size() * 4;
    ENSURE(tiles, nb_t); ENSURE(imgs, nb_i); ENSURE(seg_tile, nb_s);
    if (ensure_pin(ctx, ctx->pin_a, nb_t + nb_i + nb_s)) return 1;
    uint8_t* h = (uint8_t*)ctx->pin_a.p;
    memcpy(h, P.tiles.data(), nb_t); memcpy(h + nb_t, P.imgs.data(), nb_i); memcpy(h + nb_t + nb_i, P.seg_tile.data(), nb_s);
    CK(cudaMemcpyAsync(ctx->tiles.p, h, nb_t, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->imgs.p, h + nb_t, nb_i, cudaMemcpyHostToDevice, ctx->stream));
    if (nb_s) CK(cudaMemcpyAsync(ctx->seg_tile.p, h + nb_t + nb_i, nb_s, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Level 2 host side
// ------------------------------------------------------------------------------------------------
// Shared memory per entropy-block CTA = cum[] + tables + word ring.  Tables are sized per launch so that every
// chain of a frame is resident at once (one level: 4 B x 2^PROB_BITS; two levels: 1 KiB + 2^PROB_BITS bytes).
constexpr uint32_t lat_smem(uint32_t lut_bytes) { return LAT_CUM_WORDS * 4 + lut_bytes + LAT_RING_WORDS * 4; }
constexpr uint32_t LUT_ONE_12 = 4u << 12, LUT_ONE_14 = 4u << 14, LUT_TWO_12 = 1024 + (1u << 12), LUT_TWO_14 = 1024 + (1u << 14), LUT_TWO_15 = 1024 + (1u << 15);

// classification, RGB front end (contexts + value streams), grey candidates, backward rANS, size decisions
static int m2_encode_tiles(xpngb_ctx* ctx, const Plan& P, uint32_t ntiles, uint32_t nseg) {
    const TileDesc* d_tiles = (const TileDesc*)ctx->tiles.p;
    const uint32_t* d_seg_tile = (const uint32_t*)ctx->seg_tile.p;
    ENSURE(tclass, ntiles); ENSURE(skip, ntiles); ENSURE(tabs, (size_t)ntiles * 17 * TAB_WORDS * 4);
    ENSURE(vplace, nseg * sizeof(SegPlace)); ENSURE(vcnt, (size_t)nseg * 9 * 2);
    (void)P;
    LAUNCH(k_m2_classify, ntiles, 256, 0, d_tiles, (const ImageDesc*)ctx->imgs.p, (uint8_t*)ctx->tclass.p);
    LAUNCH(k_m2_skipmask, (ntiles + 255) / 256, 256, 0, (const uint8_t*)ctx->tclass.p, (uint8_t*)ctx->skip.p, ntiles);
    FrontArgs fa{ d_tiles, d_seg_tile, nullptr, (const uint32_t*)ctx->costs.p, (const uint8_t*)ctx->skip.p, (SegInfo*)ctx->seginfo.p,
                  (uint8_t*)ctx->sym_area.p, (uint8_t*)ctx->bits_area.p, nullptr, (uint32_t*)ctx->hist.p, (uint16_t*)ctx->vcnt.p, 0u };
    LAUNCH(k_front2<2>, nseg, FRONT_THREADS, 0, fa);           // level 2 codes RGB tiles only
    fa.rgba_only = 1;
    if (P.any_wide) LAUNCH(k_front<2>, nseg, FRONT_THREADS, 0, fa);
    TileScanArgs ta{ d_tiles, (const SegInfo*)ctx->seginfo.p, (const uint32_t*)ctx->costs.p, (const uint16_t*)ctx->vcnt.p,
                     (SegPlace*)ctx->place.p, (SegPlace*)ctx->vplace.p, (uint32_t*)ctx->hist.p, (TileState*)ctx->state.p,
                     (const uint8_t*)ctx->skip.p, ntiles };
    LAUNCH_HI(k_tile_scan<2>, (ntiles + 3) / 4, 128, 0, ta);
    CompactArgs ca{ d_tiles, d_seg_tile, (const SegInfo*)ctx->seginfo.p, (const SegPlace*)ctx->place.p, (const SegPlace*)ctx->vplace.p,
                    (const uint16_t*)ctx->vcnt.p, (const TileState*)ctx->state.p, (const uint8_t*)ctx->sym_area.p,
                    (const uint8_t*)ctx->bits_area.p, (uint8_t*)ctx->streams.p, (const uint8_t*)ctx->skip.p };
    LAUNCH(k_compact<2>, nseg, 256, 0, ca);
    LAUNCH(k_m2_grey_front, nseg, 256, 0, d_tiles, d_seg_tile, (const uint8_t*)ctx->tclass.p, (uint8_t*)ctx->streams.p, (uint32_t*)ctx->hist.p);
    RansV1Args ra{ d_tiles, (TileState*)ctx->state.p, (const uint32_t*)ctx->hist.p, (const uint8_t*)ctx->tclass.p,
                   (const uint8_t*)ctx->streams.p, (uint8_t*)ctx->blocks.p, (uint32_t*)ctx->tabs.p, ntiles, 0, 17, 0, 0 };
    auto k_rans_v1_pair_16 = k_rans_v1_pair<16>; auto k_rans_v1_pair_256 = k_rans_v1_pair<256>;
    const uint32_t ecap = 17u * ntiles;
    // blocks by decreasing length, one list per table size (enc_order.cuh)
    ENSURE(eord, (size_t)(2 * ecap + 2) * 4);
    uint32_t* eo = (uint32_t*)ctx->eord.p;
    LAUNCH_HI(k_enc_order, 1, 1024, 0, EncOrderArgs{ d_tiles, (const TileState*)ctx->state.p, (const uint8_t*)ctx->tclass.p, ntiles, 2u, eo + 2, eo, ecap });
    ra.order = eo + 2; ra.total = eo;
    // alphabets above 16 symbols and the grey candidates go to a side stream that forks BEFORE the main launch but is
    // fed AFTER it: the small-alphabet kernel holds the longest chains, and in a batch its CTAs must be placed first
    // (the 98 KiB CTAs of the other kernel would otherwise take the shared memory and delay them)
    FORK_SIDE(0);
    BACK_TO_MAIN();
    LAUNCH_HI(k_rans_v1_pair_16, (17 * ntiles + PAIR_BLK - 1) / PAIR_BLK, 32, 17 * PAIR_BLK * 24, ra);
    ctx->cur = ctx->side[0];
    RansV1Args rb = ra; rb.c0 = 9; rb.nc = 8; rb.nmin = 16;
    rb.order = ra.order + ecap; rb.total = ra.total + 1;
    LAUNCH_HI(k_rans_v1_pair_256, (8 * ntiles + PAIR_BLK - 1) / PAIR_BLK, 32, 257 * PAIR_BLK * 24, rb);
    rb.c0 = 0; rb.nc = 4; rb.nmin = 0; rb.grey = 1; rb.order = nullptr; rb.total = nullptr;
    LAUNCH_HI(k_rans_v1_pair_256, (4 * ntiles + PAIR_BLK - 1) / PAIR_BLK, 32, 257 * PAIR_BLK * 24, rb);
    JOIN_SIDE(0);
    LAUNCH_HI(k_m2_finish, (ntiles + 127) / 128, 128, 0, d_tiles, (const uint8_t*)ctx->tclass.p, (TileState*)ctx->state.p, ntiles);
    return 0;
}
// CTAs per tile for the assembly kernels: a single frame has fewer tiles than SMs, so each tile's copies are sliced
static unsigned assemble_split(uint32_t ntiles) { const uint32_t y = 592u / (ntiles ? ntiles : 1u); return y < 1u ? 1u : (y > 8u ? 8u : y); }
static int m2_assemble(xpngb_ctx* ctx, const AssembleArgs& aa, uint32_t ntiles) {
    AssembleM2Args ma{ aa, (const uint8_t*)ctx->tclass.p, (const uint32_t*)ctx->tabs.p, (const uint8_t*)ctx->streams.p };
    LAUNCH(k_assemble_m2, dim3(ntiles, assemble_split(ntiles)), 256, 0, ma);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Context and lanes
// ------------------------------------------------------------------------------------------------
static void lane_free(xpngb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int k = 0; k < xpngb_ctx::NSIDE; k++) if (ctx->side[k]) cudaStreamSynchronize(ctx->side[k]);
    DevBuf* all[] = { &ctx->pixels, &ctx->norm, &ctx->files, &ctx->arena, &ctx->tiles, &ctx->imgs, &ctx->seg_tile, &ctx->costs,
                      &ctx->hist, &ctx->seginfo, &ctx->place, &ctx->vplace, &ctx->vcnt, &ctx->sym_area, &ctx->bits_area, &ctx->alpha,
                      &ctx->streams, &ctx->blocks, &ctx->state, &ctx->outs, &ctx->flags, &ctx->skip, &ctx->dimgs, &ctx->dtiles,
                      &ctx->plane, &ctx->nlseq, &ctx->rowcnt, &ctx->rowbits, &ctx->rows, &ctx->edge, &ctx->errflag, &ctx->hdr,
                      &ctx->offs, &ctx->m2a, &ctx->m2b, &ctx->tclass, &ctx->tabs, &ctx->ccnt, &ctx->cbit, &ctx->resv, &ctx->oriented,
                      &ctx->odesc, &ctx->pdw, &ctx->eord, &ctx->region, &ctx->crops, &ctx->orients,
                      &ctx->rdescs, &ctx->rtab, &ctx->rtmp, &ctx->tdescs, &ctx->tsrc, &ctx->cdescs,
                      &ctx->bdescs, &ctx->bscr, &ctx->adescs };
    for (DevBuf* b : all) if (b->p) cudaFree(b->p);
    if (ctx->pin_a.p) cudaFreeHost(ctx->pin_a.p);
    if (ctx->pin_b.p) cudaFreeHost(ctx->pin_b.p);
    if (ctx->pin_o.p) cudaFreeHost(ctx->pin_o.p);
    if (ctx->hi) { cudaStreamSynchronize(ctx->hi); cudaStreamDestroy(ctx->hi); }
    cudaEvent_t evs[] = { ctx->ev0, ctx->ev1, ctx->ev_fork, ctx->pe0, ctx->pe1, ctx->ev_done, ctx->ev_hi };
    for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
    for (int k = 0; k < xpngb_ctx::NSIDE; k++) { if (ctx->ev_join[k]) cudaEventDestroy(ctx->ev_join[k]); if (ctx->side[k]) cudaStreamDestroy(ctx->side[k]); }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// A lane: streams, events and (empty, grow-only) scratch.  root == nullptr creates the root lane.
static xpngb_ctx* lane_new(int device, xpngb_ctx* root) {
    xpngb_ctx* ctx = new xpngb_ctx();
    ctx->device = device; ctx->root = root ? root : ctx;
    bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_done, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_hi, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreate(&ctx->ev0) == cudaSuccess && cudaEventCreate(&ctx->ev1) == cudaSuccess &&
              cudaEventCreate(&ctx->pe0) == cudaSuccess && cudaEventCreate(&ctx->pe1) == cudaSuccess;
    for (int k = 0; ok && k < xpngb_ctx::NSIDE; k++)   // side streams are created on first use (side_of): the device has at most
        ok = cudaEventCreateWithFlags(&ctx->ev_join[k], cudaEventDisableTiming) == cudaSuccess;   // 32 hardware queues, unused streams would alias used ones
    if (!ok) { lane_free(ctx); return nullptr; }
    ctx->cur = ctx->stream;
    return ctx;
}
// Lane i of a context (0 = the root itself).
static xpngb_ctx* lane_get(xpngb_ctx* root, uint32_t i) {
    if (i == 0) return root;
    while (root->lanes.size() < i) {
        xpngb_ctx* l = lane_new(root->device, root);
        if (!l) return nullptr;
        root->lanes.push_back(l);
        l->lane_id = (int)root->lanes.size();
    }
    return root->lanes[i - 1];
}

extern "C" int xpngb_create(xpngb_ctx** out, int device) {
    if (!out) return 1;
    *out = nullptr;
    // A batch call keeps up to pipe_lanes x 3 streams busy: hosts that code batches export CUDA_DEVICE_MAX_CONNECTIONS=32
    // before their first CUDA call (INTEGRATION.md 8; the driver's default of 8 hardware queues makes the streams of a call
    // wait on each other).  It is not forced here: 32 queues add ~2.5 s to every process start, which a one-image CLI run
    // should not pay (tools/ctx_time.py).
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return 1;
    if (cudaSetDevice(device) != cudaSuccess) return 1;
    xpngb_ctx* ctx = lane_new(device, nullptr);
    if (!ctx) return 1;
    if (const char* e = getenv("XPNGB_PROFILE")) ctx->profile = atoi(e) == 3 ? 3 : (atoi(e) ? 2 : 0);
    if (const char* e = getenv("XPNGB_CHUNK_MPIX")) { const long v = atol(e); if (v > 0) ctx->max_chunk_px = (uint64_t)v << 20; }
    if (const char* e = getenv("XPNGB_PIPE_LANES")) { const long v = atol(e); if (v > 0 && v <= 64) ctx->pipe_lanes = (uint32_t)v; }
    if (const char* e = getenv("XPNGB_PIPE_MIN_MPIX")) { const long v = atol(e); if (v > 0) ctx->pipe_min_px = (uint64_t)v << 20; }
    if (const char* e = getenv("XPNGB_LAT_MAX_BLOCKS")) ctx->lat_max_blocks = (uint32_t)atol(e);
    if (const char* e = getenv("XPNGB_S16_LAT_MAX_TILES")) ctx->s16_lat_max_tiles = (uint32_t)atol(e);
    if (const char* e = getenv("XPNGB_V2_DIRECT_MAX_TILES")) ctx->v2_direct_max_tiles = (uint32_t)atol(e);
    if (const char* e = getenv("XPNGB_WALK")) ctx->walk_ring = !strcmp(e, "ring");
    if (const char* e = getenv("XPNGB_DIRECT_MAX_TILES")) ctx->direct_max_tiles = (uint32_t)atol(e);
    { auto p = k_rans_v2_pair<256>; cudaFuncSetAttribute(p, cudaFuncAttributeMaxDynamicSharedMemorySize, 257 * PAIR_BLK * 24); }
    { auto p = k_rans_v1_pair<256>; cudaFuncSetAttribute(p, cudaFuncAttributeMaxDynamicSharedMemorySize, 257 * PAIR_BLK * 24); }
    cudaFuncSetAttribute(k_dec_unpredict_rows<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 2 * 32 * UNR_PITCH);
    cudaFuncSetAttribute(k_dec_unpredict_rows<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 2 * 32 * UNR_PITCH);
    cudaFuncSetAttribute(k_dec_walk_smem<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (WALK_SMEM_MAX_SYMS / 8 + 32) * 4);
    cudaFuncSetAttribute(k_dec_rans_v1_lat, cudaFuncAttributeMaxDynamicSharedMemorySize, lat_smem(LUT_ONE_14));
    { auto p = k_dec_rans_pair<1, 0>; cudaFuncSetAttribute(p, cudaFuncAttributeMaxDynamicSharedMemorySize, PD_WARPS * PD_BIG_BYTES); }
    { auto p = k_dec_rans_pair<2, 0>; cudaFuncSetAttribute(p, cudaFuncAttributeMaxDynamicSharedMemorySize, PD_WARPS * PD_BIG_BYTES); }
    *out = ctx;
    return 0;
}

extern "C" void xpngb_destroy(xpngb_ctx* ctx) {
    if (!ctx) return;
    for (xpngb_ctx* l : ctx->lanes) lane_free(l);
    ctx->lanes.clear();
    lane_free(ctx);
}

extern "C" const char* xpngb_last_error(const xpngb_ctx* ctx) { return ctx ? ctx->err : "no context"; }
extern "C" float xpngb_last_kernel_ms(const xpngb_ctx* ctx) { return ctx ? ctx->last_ms : 0.f; }
extern "C" uint32_t xpngb_last_launches(const xpngb_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" uint64_t xpngb_last_tiles(const xpngb_ctx* ctx) { return ctx ? ctx->decoded_tiles : 0; }
extern "C" void* xpngb_stream(const xpngb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

extern "C" void xpngb_profile(xpngb_ctx* ctx, int on) { if (ctx) { ctx->profile = on == 3 ? 3 : (on ? (ctx->profile == 2 ? 2 : 1) : 0); ctx->prof.clear(); } }
extern "C" uint32_t xpngb_profile_report(const xpngb_ctx* ctx, char* buf, uint32_t cap) {
    uint32_t n = 0;
    if (!ctx || !buf || !cap) return 0;
    buf[0] = 0;
    for (const auto& r : ctx->prof) {
        const int k = snprintf(buf + n, cap - n, "%s %.6f %u\n", r.name, r.ms, r.count);
        if (k < 0 || (uint32_t)k >= cap - n) break;
        n += (uint32_t)k;
    }
    return n;
}

extern "C" uint64_t xpngb_encode_bound(const xpngb_image* imgs, uint32_t n) {
    uint64_t t = 0;
    for (uint32_t i = 0; i < n; i++) t += (8 + imgs[i].w * imgs[i].h * (3 + (imgs[i].A ? 1 : 0)) + 15) & ~15ull;
    return t;
}

extern "C" int xpngb_peek(const void* file, uint64_t size, xpngb_image* img) {
    if (!file || !img || size < 8) return 1;
    uint32_t h[2]; memcpy(h, file, 8);
    img->w = (h[0] & 0xFFFFFFu) + 1; img->h = (h[1] & 0xFFFFFFu) + 1; img->A = (h[1] >> 24) & 1; img->mode = h[0] >> 24;
    return !(img->mode == 1 || img->mode == 2 || img->mode == 7);   // libxpng.c:972
}

// Cut n images into chunks of whole images: at most pipe_lanes chunks of roughly equal pixel count, none below
// pipe_min_px (so small calls stay one chunk) and none above max_chunk_px (scratch bound).  Returns the chunk starts + n.
// first (may be null): a chunk may start at image i only where first[i] is set.
static std::vector<uint32_t> cut_chunks(const xpngb_ctx* ctx, const xpngb_image* imgs, uint32_t n, const uint8_t* first = nullptr) {
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) total += imgs[i].w * imgs[i].h;
    uint64_t want = (total + ctx->pipe_lanes - 1) / ctx->pipe_lanes;
    if (want < ctx->pipe_min_px) want = ctx->pipe_min_px;
    if (want > ctx->max_chunk_px) want = ctx->max_chunk_px;
    // k chunks of equal share: chunk c ends with the image that brings the running pixel count to (c + 1) / k of the total.
    // (Cutting whenever `want` pixels are exceeded leaves a small extra chunk when the images do not divide evenly, and a
    // chunk beyond the lanes waits for a lane: a whole chain latency for a handful of images.)
    uint64_t k = (total + want - 1) / want;
    if (k < 1) k = 1;
    if (k > n) k = n;
    std::vector<uint32_t> cuts{ 0 };
    uint64_t px = 0, c = 1;
    for (uint32_t i = 0; i < n && c < k; i++) {
        px += imgs[i].w * imgs[i].h;
        typedef unsigned __int128 u128;   // w, h <= 2^24 each: the products exceed 64 bits for absurd batches only, but must not wrap
        if ((u128)px * k >= (u128)c * total && i + 1 < n && (!first || first[i + 1])) {
            cuts.push_back(i + 1);
            while (c < k && (u128)px * k >= (u128)c * total) c++;
        }
    }
    cuts.push_back(n);
    return cuts;
}

// ------------------------------------------------------------------------------------------------
// Encode
// ------------------------------------------------------------------------------------------------
// Whole-image single colour at level 2 (libxpng.c:741-753), decided on the device for RGB batches so that the host
// never waits for the scan.
__global__ void k_apply_scan(ImageDesc* imgs, const uint32_t* flags, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && imgs[i].mode == 2 && !(flags[i] & SCAN_NOT_SINGLE)) imgs[i].mode = 2 | 0x100;
}

// One chunk in flight on a lane: what the host needs to finish it.
struct EncChunk {
    xpngb_ctx* lane = nullptr;
    xpngb_image* imgs = nullptr; uint32_t n = 0;
    uint32_t first = 0; const uint32_t* index = nullptr;   // caller's index of imgs[i]: index[i], or first + i (error messages)
    uint64_t* out_offsets = nullptr; uint64_t* out_sizes = nullptr;
    std::vector<uint32_t> pxsz;
    uint64_t out_base = 0, out_end = 0;     // region of the device arena: [out_base, out_end) is this chunk's bound, files are packed from out_base
    bool finished = false; uint64_t used_end = 0;
};

static int encode_finish(xpngb_ctx* ctx, EncChunk& C);

// Launch everything for one chunk on lane `ctx`; nothing here waits for the device unless the chunk holds RGBA images
// (alpha normalisation changes the pixel size, which the tile plan depends on).
static int encode_issue(xpngb_ctx* ctx, int level, const uint8_t* dpix, uint8_t* dout, EncChunk& C) {
    xpngb_image* imgs = C.imgs; const uint32_t n = C.n;
    ctx->cur = ctx->stream;
    bool any_rgba = false;
    for (uint32_t i = 0; i < n; i++) any_rgba |= imgs[i].A != 0;
    std::vector<uint32_t> flags(n, SCAN_NOT_SINGLE);
    std::vector<uint64_t> addr(n);
    std::vector<uint32_t>& pxsz = C.pxsz; pxsz.resize(n);
    for (uint32_t i = 0; i < n; i++) { addr[i] = (uint64_t)(dpix + imgs[i].offset); pxsz[i] = imgs[i].A ? 4 : 3; }
    const unsigned scan_chunks = n >= 148 ? 8u : (1184u / n > 592u ? 592u : 1184u / n);   // ~8 CTAs per SM over the whole chunk
    if (any_rgba) {
        // ---- normalisation / whole-image scans: the one place where the host waits inside a chunk
        std::vector<ImageDesc> S(n);
        for (uint32_t i = 0; i < n; i++) {
            ImageDesc I{}; I.px_off = addr[i]; I.w = (uint32_t)imgs[i].w; I.h = (uint32_t)imgs[i].h; I.pxsz = pxsz[i];
            I.raw_size = imgs[i].w * imgs[i].h * pxsz[i];
            S[i] = I;
        }
        const size_t nb = n * sizeof(ImageDesc);
        ENSURE(imgs, nb); ENSURE(flags, n * 4);
        if (ensure_pin(ctx, ctx->pin_a, nb)) return 1;
        memcpy(ctx->pin_a.p, S.data(), nb);
        CK(cudaMemcpyAsync(ctx->imgs.p, ctx->pin_a.p, nb, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemsetAsync(ctx->flags.p, 0, n * 4, ctx->stream));
        LAUNCH(k_image_scan, dim3(scan_chunks, n), 256, 0, (const ImageDesc*)ctx->imgs.p, (uint32_t*)ctx->flags.p);
        CK(cudaMemcpyAsync(flags.data(), ctx->flags.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        // apply normalisation (libxpng.c:688-721)
        uint64_t need = 0;
        for (uint32_t i = 0; i < n; i++) if (imgs[i].A && ((flags[i] & SCAN_DIRTY) || !(flags[i] & SCAN_TRANSLUCENT)))
            need += (imgs[i].w * imgs[i].h * 4 + 15) & ~15ull;
        if (need) {
            ENSURE(norm, need);
            uint64_t o = 0;
            for (uint32_t i = 0; i < n; i++) {
                if (!imgs[i].A) continue;
                const uint64_t npx = imgs[i].w * imgs[i].h;
                uint8_t* dst = (uint8_t*)ctx->norm.p + o;
                const unsigned grid = (unsigned)((npx + 1023) / 1024 > 1184 ? 1184 : (npx + 1023) / 1024);
                if (flags[i] & SCAN_DIRTY) LAUNCH(k_alpha_zero, grid, 256, 0, (const uint32_t*)addr[i], (uint32_t*)dst, npx);
                else if (!(flags[i] & SCAN_TRANSLUCENT)) { LAUNCH(k_alpha_strip, grid, 256, 0, (const uint32_t*)addr[i], dst, npx); pxsz[i] = 3; }
                else continue;
                addr[i] = (uint64_t)dst; o += (npx * 4 + 15) & ~15ull;
            }
        }
    }
    // ---- effective level per image (libxpng.c:735, :741-755).  Without RGBA images the single-colour test of level 2
    // is applied on the device (k_apply_scan); the host only needs to know that level-2 work exists.
    std::vector<uint32_t> mode(n);
    bool any1 = false, any2 = false;
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t s = imgs[i].w * imgs[i].h * pxsz[i];
        uint32_t m = (uint32_t)level;
        if (s <= 4) m = 7;
        if (m == 2 && any_rgba && !(flags[i] & SCAN_NOT_SINGLE)) m = 2 | 0x100;
        else if (m == 2 && pxsz[i] == 4) m = 1;
        if ((m == 1) && pxsz[i] == 4 && (imgs[i].w < 4 || imgs[i].h < 4))
            FAIL("image %u: RGBA tiles thinner than 4 pixels are not encodable at level 1/2 (the reference crashes here)",
                 C.index ? C.index[i] : C.first + i);
        mode[i] = m; any1 |= m == 1; any2 |= m == 2;
    }
    if (any1 && any2) {
        // level 2 with some images that keep alpha (coded at level 1, libxpng.c:755): the chunk is regrouped into the two
        // families and each family is encoded in ONE pass (files of a family are adjacent in the arena; the offset table,
        // not the arena order, is the contract).  Only chunks with RGBA images get here, and they have waited already.
        uint64_t base = C.out_base;
        for (int fam = 0; fam < 2; fam++) {
            std::vector<uint32_t> idx;
            for (uint32_t i = 0; i < n; i++) if ((mode[i] == 1) == (fam == 0)) idx.push_back(i);
            if (idx.empty()) continue;
            std::vector<xpngb_image> sub(idx.size());
            std::vector<uint64_t> so(idx.size()), ss(idx.size());
            std::vector<uint32_t> caller(idx.size());
            for (size_t k = 0; k < idx.size(); k++) { sub[k] = imgs[idx[k]]; caller[k] = C.index ? C.index[idx[k]] : C.first + idx[k]; }
            EncChunk S; S.lane = ctx; S.imgs = sub.data(); S.n = (uint32_t)idx.size(); S.out_offsets = so.data(); S.out_sizes = ss.data();
            S.index = caller.data();
            S.out_base = base; S.out_end = C.out_end;
            if (encode_issue(ctx, fam == 0 ? 1 : 2, dpix, dout, S) || encode_finish(ctx, S)) return 1;
            base = S.used_end;
            for (size_t k = 0; k < idx.size(); k++) { imgs[idx[k]] = sub[k]; C.out_offsets[idx[k]] = so[k]; C.out_sizes[idx[k]] = ss[k]; }
        }
        C.finished = true; C.used_end = base;
        CK(cudaEventRecord(ctx->ev_done, ctx->stream));
        return 0;
    }
    // ---- plan
    Plan P;
    const int sfac = any2 ? 4 : 1, bfac = any2 ? 8 : 4;
    for (uint32_t i = 0; i < n; i++) plan_image(P, addr[i], imgs[i].w, imgs[i].h, pxsz[i], mode[i], sfac, bfac);
    if (P.tiles.size() > (1u << 24) || P.seg_tile.size() > (1u << 28)) FAIL("too many tiles for one chunk (%zu)", P.tiles.size());
    const uint32_t ntiles = (uint32_t)P.tiles.size(), nseg = (uint32_t)P.seg_tile.size();
    if (upload_plan(ctx, P)) return 1;
    ENSURE(outs, n * sizeof(ImageOut)); ENSURE(state, ntiles * sizeof(TileState));
    CK(cudaMemsetAsync(ctx->state.p, 0, ntiles * sizeof(TileState), ctx->stream));
    const TileDesc* d_tiles = (const TileDesc*)ctx->tiles.p;
    const ImageDesc* d_imgs = (const ImageDesc*)ctx->imgs.p;
    const uint32_t* d_seg_tile = (const uint32_t*)ctx->seg_tile.p;
    if (any2 && !any_rgba) {
        ENSURE(flags, n * 4);
        CK(cudaMemsetAsync(ctx->flags.p, 0, n * 4, ctx->stream));
        LAUNCH(k_image_scan, dim3(scan_chunks, n), 256, 0, d_imgs, (uint32_t*)ctx->flags.p);
        LAUNCH(k_apply_scan, (n + 127) / 128, 128, 0, (ImageDesc*)ctx->imgs.p, (const uint32_t*)ctx->flags.p, n);
    }

    if (any1 || any2) {
        const int hstride = any2 ? HIST_STRIDE_M2 : HIST_STRIDE_M1;
        ENSURE(costs, ntiles * 16); ENSURE(hist, (size_t)ntiles * hstride * 4); ENSURE(seginfo, nseg * sizeof(SegInfo));
        ENSURE(place, nseg * sizeof(SegPlace)); ENSURE(sym_area, (size_t)nseg * SEG); ENSURE(bits_area, (size_t)nseg * SEG_BITS_BYTES + 64);
        ENSURE(streams, P.str_total); ENSURE(blocks, P.blk_total);
        if (P.any_rgba) ENSURE(alpha, P.px_total);
        CK(cudaMemsetAsync(ctx->costs.p, 0, ntiles * 16, ctx->stream));
        CK(cudaMemsetAsync(ctx->hist.p, 0, (size_t)ntiles * hstride * 4, ctx->stream));
        LAUNCH(k_predictor_cost, dim3(ntiles, PP_SPLIT), 256, 0, d_tiles, (const uint8_t*)nullptr, (uint32_t*)ctx->costs.p);
    }
    if (any1) {
        FrontArgs fa{ d_tiles, d_seg_tile, nullptr, (const uint32_t*)ctx->costs.p, nullptr, (SegInfo*)ctx->seginfo.p,
                      (uint8_t*)ctx->sym_area.p, (uint8_t*)ctx->bits_area.p, (uint8_t*)ctx->alpha.p, (uint32_t*)ctx->hist.p, nullptr, 0u };
        bool any_rgb = false;
        for (uint32_t i = 0; i < n; i++) any_rgb |= pxsz[i] == 3 && mode[i] == 1;
        if (any_rgb) LAUNCH(k_front2<1>, nseg, FRONT_THREADS, 0, fa);
        fa.rgba_only = 1;
        if (P.any_rgba || P.any_wide) LAUNCH(k_front<1>, nseg, FRONT_THREADS, 0, fa);
        TileScanArgs ta{ d_tiles, (const SegInfo*)ctx->seginfo.p, (const uint32_t*)ctx->costs.p, nullptr, (SegPlace*)ctx->place.p, nullptr,
                         (uint32_t*)ctx->hist.p, (TileState*)ctx->state.p, nullptr, ntiles };
        LAUNCH_HI(k_tile_scan<1>, (ntiles + 3) / 4, 128, 0, ta);
        CompactArgs ca{ d_tiles, d_seg_tile, (const SegInfo*)ctx->seginfo.p, (const SegPlace*)ctx->place.p, nullptr, nullptr,
                        (const TileState*)ctx->state.p, (const uint8_t*)ctx->sym_area.p, (const uint8_t*)ctx->bits_area.p,
                        (uint8_t*)ctx->streams.p, nullptr };
        LAUNCH(k_compact<1>, nseg, 256, 0, ca);
        RansV2Args ra{ d_tiles, (TileState*)ctx->state.p, (uint32_t*)ctx->hist.p, (const uint8_t*)ctx->streams.p,
                       (const uint8_t*)ctx->alpha.p, (uint8_t*)ctx->blocks.p, ntiles, 0, 9 };
        auto k_rans_v2_pair_16 = k_rans_v2_pair<16>; auto k_rans_v2_pair_256 = k_rans_v2_pair<256>;
        const uint32_t ecap = 10u * ntiles;
        // blocks by decreasing length (enc_order.cuh)
        ENSURE(eord, (size_t)(2 * ecap + 2) * 4);
        uint32_t* eo = (uint32_t*)ctx->eord.p;
        LAUNCH_HI(k_enc_order, 1, 1024, 0, EncOrderArgs{ d_tiles, (const TileState*)ctx->state.p, nullptr, ntiles, 1u, eo + 2, eo, ecap });
        ra.order = eo + 2; ra.total = eo;
        if (P.any_rgba) {                          // the alpha blocks are independent of the context blocks: side stream
            FORK_SIDE(0);                          // forks before, is fed after the main launch (see m2_encode_tiles)
            BACK_TO_MAIN();
        }
        LAUNCH_HI(k_rans_v2_pair_16, (9 * ntiles + PAIR_BLK - 1) / PAIR_BLK, 32, 17 * PAIR_BLK * 24, ra);
        if (P.any_rgba) {
            RansV2Args rb = ra; rb.c0 = 9; rb.nc = 1;
            rb.order = ra.order + ecap; rb.total = ra.total + 1;
            ctx->cur = ctx->side[0];
            LAUNCH_HI(k_rans_v2_pair_256, (ntiles + PAIR_BLK - 1) / PAIR_BLK, 32, 257 * PAIR_BLK * 24, rb);
            JOIN_SIDE(0);
        }
    }
    if (any2) {
        if (m2_encode_tiles(ctx, P, ntiles, nseg)) return 1;
    }
    LAUNCH_HI(k_image_sizes, (n + 127) / 128, 128, 0, d_imgs, d_tiles, (TileState*)ctx->state.p, (ImageOut*)ctx->outs.p, n);
    LAUNCH_HI(k_image_offsets, 1, 1, 0, (ImageOut*)ctx->outs.p, n, C.out_base);
    {
        AssembleArgs aa{ d_imgs, d_tiles, (const TileState*)ctx->state.p, (const ImageOut*)ctx->outs.p, (const SegInfo*)ctx->seginfo.p,
                         (const SegPlace*)ctx->place.p, nullptr, (const uint8_t*)ctx->bits_area.p, (const uint8_t*)ctx->blocks.p, dout };
        if (any2) { if (m2_assemble(ctx, aa, ntiles)) return 1; }
        else LAUNCH(k_assemble_m1, dim3(ntiles, assemble_split(ntiles)), 256, 0, aa);
    }
    if (ensure_pin(ctx, ctx->pin_b, n * sizeof(ImageOut))) return 1;
    CK(cudaMemcpyAsync(ctx->pin_b.p, ctx->outs.p, n * sizeof(ImageOut), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_done, ctx->stream));
    return 0;
}

// Wait for the chunk's size table and hand the results to the caller's arrays.
static int encode_finish(xpngb_ctx* ctx, EncChunk& C) {
    CK(cudaEventSynchronize(ctx->ev_done));
    if (C.finished) return 0;
    const ImageOut* ho = (const ImageOut*)ctx->pin_b.p;
    uint64_t end = C.out_base;
    for (uint32_t i = 0; i < C.n; i++) {
        C.out_offsets[i] = ho[i].off; C.out_sizes[i] = ho[i].size;
        C.imgs[i].A = C.pxsz[i] == 4; C.imgs[i].mode = ho[i].mode & 0xFF;
        end = ho[i].off + ((ho[i].size + 15) & ~15ull);
    }
    if (end > C.out_end) FAIL("output region too small: need %llu bytes, have %llu", (unsigned long long)(end - C.out_base), (unsigned long long)(C.out_end - C.out_base));
    C.finished = true; C.used_end = end;
    return 0;
}

extern "C" int xpngb_encode(xpngb_ctx* ctx, int level, xpngb_image* imgs, uint32_t n, const void* pixels, uint64_t pixels_size,
                            int pixels_on_device, void* out, uint64_t out_cap, int out_on_device, uint64_t* out_offsets,
                            uint64_t* out_sizes) {
    if (!ctx) return 1;
    ctx->err[0] = 0; ctx->launches = 0; ctx->last_ms = 0.f; ctx->cur = ctx->stream;
    if (!imgs || !pixels || !out || !out_offsets || !out_sizes) FAIL("null argument");
    if (!(level == 1 || level == 2 || level == 7)) FAIL("level must be 1, 2 or 7");          // libxpng.c:729
    if (n == 0) return 0;
    for (uint32_t i = 0; i < n; i++) {
        const xpngb_image& m = imgs[i];
        if (!m.w || !m.h || m.w > (1u << 24) || m.h > (1u << 24)) FAIL("image %u: bad dimensions", i);   // libxpng.c:729-730
        if (m.offset & 15) FAIL("image %u: pixel offset must be a multiple of 16", i);
        const uint64_t bytes = m.w * m.h * (3 + (m.A ? 1 : 0));   // w, h <= 2^24: no overflow
        if (bytes > pixels_size || m.offset > pixels_size - bytes) FAIL("image %u: pixels exceed the buffer", i);
    }
    CK(cudaSetDevice(ctx->device));
    const uint64_t bound = xpngb_encode_bound(imgs, n);
    if (out_on_device && out_cap < bound) FAIL("device output buffer must hold xpngb_encode_bound() = %llu bytes", (unsigned long long)bound);
    const uint8_t* dpix = (const uint8_t*)pixels;
    if (!pixels_on_device) { ENSURE(pixels, pixels_size); dpix = (const uint8_t*)ctx->pixels.p; }
    uint8_t* dout = (uint8_t*)out;
    if (!out_on_device) { ENSURE(arena, bound); dout = (uint8_t*)ctx->arena.p; }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    bool any_rgba = false;
    for (uint32_t i = 0; i < n; i++) any_rgba |= imgs[i].A != 0;
    if (level == 7 && !any_rgba) {
        // stored files need no tiles: header + copy
        if (!pixels_on_device) CK(cudaMemcpyAsync(ctx->pixels.p, pixels, pixels_size, cudaMemcpyHostToDevice, ctx->stream));
        uint64_t used = 0;
        std::vector<ImageDesc> I(n); std::vector<uint64_t> offs(n);
        for (uint32_t i = 0; i < n; i++) {
            I[i] = ImageDesc{}; I[i].px_off = (uint64_t)(dpix + imgs[i].offset); I[i].w = (uint32_t)imgs[i].w; I[i].h = (uint32_t)imgs[i].h;
            I[i].pxsz = 3; I[i].raw_size = imgs[i].w * imgs[i].h * 3;
            offs[i] = used; out_offsets[i] = used; out_sizes[i] = 8 + I[i].raw_size; used += (out_sizes[i] + 15) & ~15ull;
            imgs[i].mode = 7;
        }
        ENSURE(imgs, n * sizeof(ImageDesc)); ENSURE(offs, n * 8);
        if (ensure_pin(ctx, ctx->pin_a, n * (sizeof(ImageDesc) + 8))) return 1;
        memcpy(ctx->pin_a.p, I.data(), n * sizeof(ImageDesc)); memcpy((uint8_t*)ctx->pin_a.p + n * sizeof(ImageDesc), offs.data(), n * 8);
        CK(cudaMemcpyAsync(ctx->imgs.p, ctx->pin_a.p, n * sizeof(ImageDesc), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->offs.p, (uint8_t*)ctx->pin_a.p + n * sizeof(ImageDesc), n * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(k_store7, dim3(296, n), 256, 0, (const ImageDesc*)ctx->imgs.p, (const uint64_t*)ctx->offs.p, dout);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        if (!out_on_device) {
            if (used > out_cap) { CK(cudaStreamSynchronize(ctx->stream)); FAIL("output buffer too small: need %llu bytes, have %llu", (unsigned long long)used, (unsigned long long)out_cap); }
            CK(cudaMemcpyAsync(out, dout, used, cudaMemcpyDeviceToHost, ctx->stream));
        }
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
        return 0;
    }
    // ---- chunks on lanes
    const std::vector<uint32_t> cuts = cut_chunks(ctx, imgs, n);
    const uint32_t nchunks = (uint32_t)cuts.size() - 1;
    std::vector<EncChunk> chunks(nchunks);
    uint64_t host_packed = 0;   // host output: files are packed across chunks
    int rc = 0;
    auto harvest = [&](uint32_t ci) -> int {   // finish chunk ci; host output: start its D2H copy on its lane
        EncChunk& C = chunks[ci];
        xpngb_ctx* lane = C.lane;
        if (encode_finish(lane, C)) return 1;
        if (!out_on_device) {
            const uint64_t len = C.used_end - C.out_base;
            if (host_packed + len > out_cap) FAIL("output buffer too small: need more than %llu bytes, have %llu", (unsigned long long)(host_packed + len), (unsigned long long)out_cap);
            CK(cudaMemcpyAsync((uint8_t*)out + host_packed, dout + C.out_base, len, cudaMemcpyDeviceToHost, lane->stream));
            for (uint32_t i = 0; i < C.n; i++) C.out_offsets[i] = C.out_offsets[i] - C.out_base + host_packed;
            host_packed += len;
        }
        return 0;
    };
    uint64_t region = 0;
    uint32_t harvested = 0;
    for (uint32_t ci = 0; ci < nchunks && !rc; ci++) {
        const uint32_t li = ci % ctx->pipe_lanes;
        while (!rc && ci >= ctx->pipe_lanes && harvested <= ci - ctx->pipe_lanes) rc = harvest(harvested++);   // the lane's previous chunk must be done
        if (rc) break;
        xpngb_ctx* lane = lane_get(ctx, li);
        if (!lane) { snprintf(ctx->err, sizeof ctx->err, "cannot create pipeline lane %u", li); rc = 1; break; }
        EncChunk& C = chunks[ci];
        C.lane = lane; C.imgs = imgs + cuts[ci]; C.n = cuts[ci + 1] - cuts[ci]; C.first = cuts[ci];
        C.out_offsets = out_offsets + cuts[ci]; C.out_sizes = out_sizes + cuts[ci];
        C.out_base = region; region += xpngb_encode_bound(C.imgs, C.n); C.out_end = region;
        if (lane != ctx) { if (cudaStreamWaitEvent(lane->stream, ctx->ev0, 0) != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "cudaStreamWaitEvent failed"); rc = 1; break; } }
        if (!pixels_on_device) {   // the chunk's pixel range (images of a chunk are adjacent in every sane layout; any layout is correct)
            uint64_t lo = ~0ull, hi = 0;
            for (uint32_t i = 0; i < C.n; i++) {
                const uint64_t a = C.imgs[i].offset, b = a + C.imgs[i].w * C.imgs[i].h * (3 + (C.imgs[i].A ? 1 : 0));
                if (a < lo) lo = a; if (b > hi) hi = b;
            }
            if (cudaMemcpyAsync((uint8_t*)ctx->pixels.p + lo, (const uint8_t*)pixels + lo, hi - lo, cudaMemcpyHostToDevice, lane->stream) != cudaSuccess) {
                snprintf(ctx->err, sizeof ctx->err, "host to device copy failed"); rc = 1; break;
            }
        }
        rc = encode_issue(lane, level, dpix, dout, C);
    }
    while (!rc && harvested < nchunks) rc = harvest(harvested++);
    // join: the root stream waits for every lane, so that ev1 closes the whole call
    for (uint32_t li = 1; li < ctx->pipe_lanes && li <= ctx->lanes.size(); li++) {
        xpngb_ctx* lane = ctx->lanes[li - 1];
        cudaEventRecord(lane->ev_done, lane->stream);
        cudaStreamWaitEvent(ctx->stream, lane->ev_done, 0);
    }
    cudaEventRecord(ctx->ev1, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && !rc) { snprintf(ctx->err, sizeof ctx->err, "device error: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
    if (rc) { for (xpngb_ctx* l : ctx->lanes) cudaStreamSynchronize(l->stream); return 1; }
    CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
    tl_dump(ctx, "enc");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Traversal-order operations (Mirroring_and_Rotating/tool.c): mirror / quarter-turn n pixmaps
// ------------------------------------------------------------------------------------------------
// The w x h source rectangle at src (rows src_pitch bytes apart) turned by op into packed rows at dst; *ctas: CTAs of the
// launch so far (k_orient runs one per 64 x 64 patch).  False when the launch would exceed the grid limit.
static bool orient_desc(OrientDesc& d, uint64_t src, uint64_t src_pitch, uint64_t dst, uint64_t w, uint64_t h, uint32_t pxsz,
                        int op, uint64_t* ctas) {
    d.src = src; d.dst = dst; d.src_pitch = src_pitch;
    d.w = (uint32_t)w; d.h = (uint32_t)h; d.pxsz = pxsz; d.op = (uint32_t)op;
    d.tiles_x = (d.w + ORI_T - 1) / ORI_T; d.first_cta = (uint32_t)*ctas;
    *ctas += (uint64_t)d.tiles_x * ((d.h + ORI_T - 1) / ORI_T);
    return *ctas <= 0x7FFFFFFFull;
}

static int orient_launch(xpngb_ctx* ctx, int op, xpngb_image* imgs, uint32_t n, const uint8_t* dsrc, uint8_t* ddst) {
    std::vector<OrientDesc> D(n);
    uint64_t ctas = 0;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t pxsz = imgs[i].A ? 4 : 3;
        if (!orient_desc(D[i], (uint64_t)(dsrc + imgs[i].offset), imgs[i].w * pxsz, (uint64_t)(ddst + imgs[i].offset), imgs[i].w,
                         imgs[i].h, pxsz, op, &ctas))
            FAIL("too many pixels for one orientation launch");
    }
    const size_t nb = n * sizeof(OrientDesc);
    ENSURE(odesc, nb);
    if (ensure_pin(ctx, ctx->pin_o, nb)) return 1;
    memcpy(ctx->pin_o.p, D.data(), nb);
    CK(cudaMemcpyAsync(ctx->odesc.p, ctx->pin_o.p, nb, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_orient, (unsigned)ctas, 256, 0, (const OrientDesc*)ctx->odesc.p, n);
    if (op == OP_R90 || op == OP_R270) for (uint32_t i = 0; i < n; i++) { const uint64_t t = imgs[i].w; imgs[i].w = imgs[i].h; imgs[i].h = t; }
    return 0;
}

static int orient_check(xpngb_ctx* ctx, int op, const xpngb_image* imgs, uint32_t n, uint64_t size) {
    if (op < OP_R90 || op > OP_TR) FAIL("unknown orientation op %d", op);
    for (uint32_t i = 0; i < n; i++) {
        const xpngb_image& m = imgs[i];
        if (!m.w || !m.h || m.w > (1u << 24) || m.h > (1u << 24)) FAIL("image %u: bad dimensions", i);
        if (m.offset & 15) FAIL("image %u: pixel offset must be a multiple of 16", i);
        const uint64_t bytes = m.w * m.h * (3 + (m.A ? 1 : 0));
        if (bytes > size || m.offset > size - bytes) FAIL("image %u: pixels exceed the buffer", i);
    }
    return 0;
}

extern "C" int xpngb_transform(xpngb_ctx* ctx, int op, xpngb_image* imgs, uint32_t n, const void* src, uint64_t size, int src_on_device,
                               void* dst, int dst_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0; ctx->launches = 0; ctx->last_ms = 0.f; ctx->cur = ctx->stream;
    if (!imgs || !src || !dst) FAIL("null argument");
    if (src == dst) FAIL("in-place orientation is not supported");
    if (!src_on_device == !dst_on_device) {   // same side: the two byte ranges must be disjoint
        const uintptr_t a = (uintptr_t)src, b = (uintptr_t)dst;
        if (a < b + size && b < a + size) FAIL("source and destination pixel buffers overlap");
    }
    if (orient_check(ctx, op, imgs, n, size)) return 1;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const uint8_t* dsrc = (const uint8_t*)src;
    if (!src_on_device) {
        ENSURE(pixels, size);
        CK(cudaMemcpyAsync(ctx->pixels.p, src, size, cudaMemcpyHostToDevice, ctx->stream));
        dsrc = (const uint8_t*)ctx->pixels.p;
    }
    uint8_t* ddst = (uint8_t*)dst;
    if (!dst_on_device) { ENSURE(oriented, size); ddst = (uint8_t*)ctx->oriented.p; }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (orient_launch(ctx, op, imgs, n, dsrc, ddst)) return 1;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (!dst_on_device) CK(cudaMemcpyAsync(dst, ddst, size, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
    return 0;
}

extern "C" int xpngb_encode_oriented(xpngb_ctx* ctx, int level, int op, xpngb_image* imgs, uint32_t n, const void* pixels,
                                     uint64_t pixels_size, int pixels_on_device, void* out, uint64_t out_cap, int out_on_device,
                                     uint64_t* out_offsets, uint64_t* out_sizes) {
    if (!ctx) return 1;
    ctx->err[0] = 0; ctx->cur = ctx->stream;
    if (!imgs || !pixels) FAIL("null argument");
    if (orient_check(ctx, op, imgs, n, pixels_size)) return 1;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const uint8_t* dsrc = (const uint8_t*)pixels;
    if (!pixels_on_device) {
        ENSURE(pixels, pixels_size);
        CK(cudaMemcpyAsync(ctx->pixels.p, pixels, pixels_size, cudaMemcpyHostToDevice, ctx->stream));
        dsrc = (const uint8_t*)ctx->pixels.p;
    }
    ENSURE(oriented, pixels_size);
    if (orient_launch(ctx, op, imgs, n, dsrc, (uint8_t*)ctx->oriented.p)) return 1;
    const uint32_t l0 = ctx->launches;
    const int rc = xpngb_encode(ctx, level, imgs, n, ctx->oriented.p, pixels_size, 1, out, out_cap, out_on_device, out_offsets, out_sizes);
    ctx->launches += l0;
    if (rc && (op == OP_R90 || op == OP_R270))   // failed: hand the descriptors back in the caller's orientation
        for (uint32_t i = 0; i < n; i++) { const uint64_t t = imgs[i].w; imgs[i].w = imgs[i].h; imgs[i].h = t; }
    return rc;
}

// ------------------------------------------------------------------------------------------------
// Decode
// ------------------------------------------------------------------------------------------------
// Work lists of the pair decoders (dec_rans_pair.cuh): two sets, one per level family present in the chunk.
static size_t pdw_bytes(uint32_t cap) { return (size_t)(2 * PD_NCLASS * PD_BUCKETS + PD_NCLASS + 5) * 4 + (size_t)PD_NCLASS * cap * 4; }
static PdWork pdw_at(void* base, uint32_t cap) {
    uint32_t* p = (uint32_t*)base;
    PdWork W; W.hist = p; W.start = p + PD_NCLASS * PD_BUCKETS; W.total = p + 2 * PD_NCLASS * PD_BUCKETS; W.order = W.total + PD_NCLASS + 5; W.cap = cap;
    return W;
}

// Bytes an entry writes at its offset: the whole image (img: w, h, A), the r->w x r->h crop, the sz->w x sz->h image or
// its win->w x win->h window, as 3 + A bytes per pixel, or with a tensor format as C elements of its dtype.  The bounds
// check and the device-to-host copy both take it from here.
static uint64_t entry_out_bytes(const xpngb_image& img, const xpngb_rect* r, const xpngb_size* sz, const xpngb_rect* win,
                                const xpngb_tensor* fmt) {
    // at most 2^24 x 2^24 (a window lies inside its size): no overflow
    const uint64_t px = win ? win->w * win->h : sz ? (uint64_t)sz->w * sz->h : r ? r->w * r->h : img.w * img.h;
    if (!fmt) return px * (3 + img.A);
    static const uint32_t elem_bytes[4] = { 1, 4, 2, 2 };   // XPNGB_DT_*
    return px * (fmt->channels == 3 ? 3 : 3 + img.A) * elem_bytes[fmt->dtype];
}

// Header checks of file i (libxpng.c:969-976) and of where its pixels go: fills imgs[i] (w, h, A, mode) and D (file,
// geometry, effective mode).  A region decode (r != nullptr) writes the r->w x r->h crop at imgs[i].offset instead of
// the whole image, a resized decode (sz != nullptr) an sz->w x sz->h image or its window win, and a tensor decode
// (fmt != nullptr) that as a tensor.  Runs for every entry of a call before anything is launched.
static int decode_check(xpngb_ctx* ctx, uint32_t i, xpngb_image& img, const uint32_t* hdr, uint64_t file_off, uint64_t file_size,
                        const xpngb_rect* r, const xpngb_size* sz, const xpngb_rect* win, const xpngb_tensor* fmt, uint64_t pixels_cap,
                        DecImage& D) {
    const uint64_t w = (hdr[0] & 0xFFFFFFu) + 1, h = (hdr[1] & 0xFFFFFFu) + 1;
    const uint32_t A = (hdr[1] >> 24) & 1, mode = hdr[0] >> 24, pxsz = 3 + A;
    if (!(mode == 1 || mode == 2 || mode == 7)) FAIL("file %u: unknown mode %u", i, mode);   // libxpng.c:972
    if (img.w && (img.w != w || img.h != h)) FAIL("file %u: header %llux%llu does not match the descriptor", i,
                                                  (unsigned long long)w, (unsigned long long)h);
    img.w = w; img.h = h; img.A = A; img.mode = mode;
    if (r && (!r->w || !r->h)) FAIL("entry %u: empty rectangle", i);
    if (r && (r->x >= w || r->w > w - r->x || r->y >= h || r->h > h - r->y))
        FAIL("entry %u: rectangle (%llu, %llu) %llux%llu is not inside the %llux%llu image", i, (unsigned long long)r->x,
             (unsigned long long)r->y, (unsigned long long)r->w, (unsigned long long)r->h, (unsigned long long)w, (unsigned long long)h);
    const uint64_t s = w * h * pxsz, out = entry_out_bytes(img, r, sz, win, fmt);
    if (img.offset & 15) FAIL("file %u: pixel offset must be a multiple of 16", i);
    if (out > pixels_cap || img.offset > pixels_cap - out) FAIL("file %u: pixels exceed the output buffer", i);
    uint32_t m = mode;
    if (mode == 7) { if (file_size < 8 + s) FAIL("file %u: truncated stored image", i); }
    else if (file_size == 11 + A && ((hdr[1] >> 24) & 2)) m = mode | 0x100;      // libxpng.c:976
    // dimensions come from an untrusted header and size every scratch buffer below: a tile is at most 666 x 666 pixels and
    // its blob at least 8 bytes, so a coded file shorter than that cannot hold the image it claims
    else if (file_size < 8 + 8 * (w * h / (666ull * 666ull))) FAIL("file %u: %llu bytes cannot hold a %llux%llu image", i,
                                                                   (unsigned long long)file_size, (unsigned long long)w, (unsigned long long)h);
    D = DecImage{};
    D.file_off = file_off; D.file_size = file_size; D.px_off = img.offset; D.w = (uint32_t)w; D.h = (uint32_t)h;
    D.pxsz = pxsz; D.mode = m;
    return 0;
}

// One entry of a region decode: the rectangle, the tiles that hold it and their union.  A resampled entry (rs) of a resized
// decode resamples its crop to `full` with `filter` and keeps the window `win` (in full's coordinates); its rectangle is
// then the span of the crop that the window's support reaches.
struct RegionSel {
    xpngb_rect rect, cover; TileGrid g; TileSel s;
    bool rs; uint32_t filter; xpngb_rect crop, win; xpngb_size full;
};
static bool whole_tiles(const RegionSel& R) {
    return R.rect.x == R.cover.x && R.rect.y == R.cover.y && R.rect.w == R.cover.w && R.rect.h == R.cover.h;
}
static uint64_t window_pitch(const xpngb_rect& cover, uint32_t pxsz) { return (cover.w * pxsz + 15) & ~15ull; }   // keeps RGB rows word-aligned (tile_pitched)
static uint64_t window_pitch(const RegionSel& R, uint32_t pxsz) { return window_pitch(R.cover, pxsz); }
// Position p of a call whose entries are ordered by file (group_entries).  n: entries decoded from one shared window, at
// its first position (0 at the others); 1 for an entry decoded as on its own (the only entry of its file, or a stored
// file).  s, cover (n > 1): the tile bounding box of the group's rectangles, and its pixels.
struct Share { uint32_t n; TileSel s; xpngb_rect cover; };
// Entry i of an oriented decode is written turned or mirrored.  TL and TR are copies in the reference: those entries are
// decoded exactly as without an op.
static bool turned(const int* ops, uint32_t i) { return ops && ops[i] != OP_TL && ops[i] != OP_TR; }
// Pillow's number of weights per output coordinate of one axis (0: the axis is not resampled, or not a filter).
static uint32_t resize_ksize(uint32_t filter, uint64_t in, uint64_t out) {
    if (in == out || resize_support(filter) == 0.0) return 0;
    const double scale = (double)in / (double)out;
    return 2 * (uint32_t)ceil(resize_support(filter) * (scale < 1.0 ? 1.0 : scale)) + 1;
}
static uint32_t resize_kx(const RegionSel& R) { return resize_ksize(R.filter, R.crop.w, R.full.w); }
static uint32_t resize_ky(const RegionSel& R) { return resize_ksize(R.filter, R.crop.h, R.full.h); }
static uint64_t resize_tab_bytes(const RegionSel& R) {
    return resize_table_bytes((uint32_t)R.win.w, resize_kx(R)) + resize_table_bytes((uint32_t)R.win.h, resize_ky(R));
}
// Scratch of resampled entry R: tables (a multiple of 8 bytes) and the first pass's rows (16-byte aligned) when both axes
// are resampled: the span's rows of window-wide pixels, or window rows of span-wide pixels when the vertical pass runs first.
static uint64_t resize_tmp_bytes(const RegionSel& R, uint32_t pxsz) {
    if (!resize_kx(R) || !resize_ky(R)) return 0;
    const uint64_t px = resize_vfirst(R.crop.w, R.crop.h, R.full.w, R.full.h) ? R.win.h * R.rect.w : R.rect.h * R.win.w;
    return (px * pxsz + 15) & ~15ull;
}
// [lo, hi): the input coordinates that the windows of output coordinates o0 .. o1 - 1 of one axis read, widened by one
// pixel on each side and clipped to [0, in), so that this plain host arithmetic needs no bit-exact agreement with the
// device's tables (windows are monotone in the output coordinate for every filter).
static void resize_span(uint32_t filter, uint64_t in, uint64_t out, uint64_t o0, uint64_t o1, uint64_t& lo, uint64_t& hi) {
    const double scale = (double)in / (double)out, support = resize_support(filter) * (scale < 1.0 ? 1.0 : scale);
    const int64_t a = (int64_t)((o0 + 0.5) * scale - support + 0.5) - 1, b = (int64_t)((o1 - 0.5) * scale + support + 0.5) + 1;
    lo = a < 0 ? 0 : (uint64_t)a;
    hi = b > (int64_t)in ? in : (uint64_t)b;
}
// The longest crop side a filter may resample.  The accumulator starts at 2^21 and adds src * k over an axis's n <= in
// taps, src in 0..255, in any order of signs; every partial sum lies within 2^21 +- 255 * sum |k|.  Each integer weight is
// its normalised weight w times 2^22, rounded by at most 1/2, so sum |k| <= 2^22 * (1 + 2 * N) + n / 2, N being the sum of
// the negative normalised weights of one output coordinate.  That stays below 2^31 while 1 + 2 * N + n / 2^23 <= 2.0058
// (2^31 is 2.0078 * 255 * 2^22, less the 2^21 start).  Box, bilinear and hamming have no negative weights (N = 0):
// n <= 2^23.  Over every in, out <= 256, where clipped windows make it largest, N is at most 0.134 for bicubic (208 -> 193)
// and 0.286 for lanczos (4 -> 5; tests/test_resampled_decode.py measures both).  So bicubic gets 2^22 (room for N up to
// 0.25) and lanczos 2^21 (room for N up to 0.375).
static uint64_t resize_side_max(uint32_t filter) { return filter == RF_LANCZOS ? 1ull << 21 : filter == RF_BICUBIC ? 1ull << 22 : 1ull << 23; }

// Pillow's box radius and weights of one axis of GaussianBlur(r), three passes: _gaussian_blur_radius and the head of
// ImagingHorizontalBoxBlur (BoxBlur.c), operation for operation in float.  r is finite, 0 < r <= XPNGB_BLUR_RADIUS_MAX
// (below it fr >= 0 and (2 ri + 1) * ww <= 2^24, so fw does not wrap; blur.cuh has the rest of the bound).
struct BlurBox { int32_t ri; uint32_t ww, fw; };
static BlurBox blur_box(float r) {
    const float sigma2 = r * r / 3.f;
    const float L = (float)sqrt((double)(sigma2 * 12.f + 1.f));
    const float l = floorf((L - 1.f) / 2.f);
    float a = (2.f * l + 1.f) * (l * (l + 1.f) - 3.f * sigma2);
    a /= 6.f * (sigma2 - (l + 1.f) * (l + 1.f));
    const float fr = l + a;
    BlurBox b;
    b.ri = (int32_t)fr;
    b.ww = (uint32_t)(16777216.f / (fr * 2.f + 1.f));
    b.fw = ((1u << 24) - (uint32_t)(b.ri * 2 + 1) * b.ww) / 2;
    return b;
}
static bool blur_on(const xpngb_blur& b) { return (float)b.radius[0] != 0.f || (float)b.radius[1] != 0.f || b.solarize; }
// ImageOps.solarize's `v < threshold` for bytes v is v < ceil(threshold), clamped to the bytes: 256 keeps them all
static uint32_t solarize_t(double threshold) {
    const double c = ceil(threshold);
    return c <= 0.0 ? 0u : c >= 256.0 ? 256u : (uint32_t)c;
}
// the op turns the entry a quarter: its output's x axis is the staged pixels' y axis
static bool quarter(const int* ops, uint32_t i) { return ops && (ops[i] == OP_R90 || ops[i] == OP_R270); }

// C's (int) of a double as Pillow's x86-64 build computes it (cvttsd2si): INT_MIN for NaN and out of range
static int32_t x86_int(double v) { return v > -2147483649.0 && v < 2147483648.0 ? (int32_t)v : INT32_MIN; }
// Geometry.c's FIX: 16.16 fixed point, FLOOR(v * 65536.0 + 0.5)
static int32_t pil_fix(double v) { const double t = v * 65536.0 + 0.5; return t < 0.0 ? x86_int(floor(t)) : x86_int(t); }
// check_fixed at the four corners of a W x H output: affine_fixed's 16.16 arithmetic can hold every source coordinate
static bool affine_fixed_ok(const double* a, double W, double H) {
    const double cx[4] = { 0.0, W, 0.0, W }, cy[4] = { 0.0, H, H, 0.0 };
    for (int k = 0; k < 4; k++)
        if (!(fabs(cx[k] * a[0] + cy[k] * a[1] + a[2]) < 32768.0 && fabs(cx[k] * a[3] + cy[k] * a[4] + a[5]) < 32768.0)) return false;
    return true;
}
constexpr uint32_t AUG_STAGES = XPNGB_AUG_STEPS_MAX + 1;   // a uint8 entry whose last step wrote its scratch gets one copy back

// Launch the decode of one chunk on lane `ctx`.  DI: the checked images of the chunk.  `lat`: warp-per-block chain
// kernels (few blocks in the whole call) instead of the pair decoders.  sel == nullptr: every tile of every image, in
// place.  Otherwise a region decode: only the tiles of sel[i].s, written in place when the rectangle is made of whole
// tiles, else into a window of the lane's region scratch from which k_crop_rows copies the rectangle; stored images
// are cropped straight out of their files.  ops (only with sel): an entry that is turned (turned()) always goes through a
// window, or for a stored image straight out of its file, and one k_orient launch writes all of them.  A resampled entry
// (sel[i].rs) also always goes through a window or its file, and is resampled and written through its op by one launch
// of each resize kernel for the chunk.  fmt (only with sel): every entry goes through a window or its
// file, a resized one is resampled without its op into the lane's tsrc scratch, and one k_to_tensor launch writes every
// entry's tensor through its op.  colors (only with sel): a coloured entry's pixels are changed in place by one
// k_color_mean and one k_color launch after the resize launches: at its uint8 output, or for a tensor entry in tsrc (a
// resized one lands there anyway, any other is copied there by k_crop_rows), from which k_to_tensor reads it.  blurs (only
// with sel): a blurred or solarized entry is staged as a coloured one is, then goes through its box passes after k_color,
// ping-ponged between its pixels and the lane's bscr scratch, one k_blur launch per pass stage of the chunk; a tensor
// entry's k_to_tensor reads whichever buffer its last pass wrote, a uint8 entry's passes end at its output.  share (only
// with sel, may be null): the entries of a group with share[i].n > 1 read one file; its first entry decodes the group's
// tile bounding box into one window, and every entry of the group goes on from there as from its own window (the others
// plan no tiles).  Never waits for the device.
static int decode_issue(xpngb_ctx* ctx, bool lat, const xpngb_image* imgs, const DecImage* DI_in, const RegionSel* sel, const Share* share,
                        const int* ops, const xpngb_tensor* fmt, const xpngb_color* colors, const xpngb_blur* blurs,
                        const xpngb_augment* augs, uint32_t n, const uint8_t* din, uint8_t* dpx, uint32_t call_tiles) {
    ctx->cur = ctx->stream;
    Plan P;
    std::vector<DecImage> DI(DI_in, DI_in + n);
    std::vector<CropDesc> crops;
    std::vector<OrientDesc> odescs;
    std::vector<ResizeDesc> rdescs;
    std::vector<TensorDesc> tdescs;
    std::vector<ColorDesc> cdescs;
    std::vector<BlurPass> bstage[BLUR_STAGES];   // the k-th pass of every blurred entry is in bstage[k]
    std::vector<AugPix> apix[AUG_STAGES];        // step k of every augmented entry, by kind: warps and SHARPNESS,
    std::vector<ColorDesc> acol[AUG_STAGES];     // BRIGHTNESS, COLOR and CONTRAST,
    std::vector<AugLut> alut[AUG_STAGES];        // and the LUT steps
    uint64_t apctas[AUG_STAGES] = {}, acctas[AUG_STAGES] = {}, amctas[AUG_STAGES] = {}, alctas[AUG_STAGES] = {}, ahctas[AUG_STAGES] = {};
    uint32_t anhist[AUG_STAGES] = {};
    uint64_t octas = 0, rcoef = 0, rh = 0, rv = 0, tctas = 0, cctas = 0, mctas = 0;
    bool any1 = false, any2 = false, any7 = false;
    for (uint32_t i = 0; i < n; i++) { any1 |= DI[i].mode == 1; any2 |= DI[i].mode == 2; any7 |= DI[i].mode == 7; }
    auto colored = [&](uint32_t i) { return colors && (colors[i].on || colors[i].gray); };
    auto blurred = [&](uint32_t i) { return blurs && blur_on(blurs[i]); };
    auto augmented = [&](uint32_t i) { return augs && augs[i].nsteps; };
    auto staged = [&](uint32_t i) { return colored(i) || blurred(i) || augmented(i); };   // needs its uint8 pixels to work on
    auto shared = [&](uint32_t i) { return share && share[i].n != 1; };                  // goes on from its group's window
    // pixels entry i writes: its resampled window, or its rectangle
    auto out_px = [&](uint32_t i) -> uint64_t { return sel[i].rs ? sel[i].win.w * sel[i].win.h : sel[i].rect.w * sel[i].rect.h; };
    // uint8 pixels of a resized or staged tensor entry, or of a blurred entry's scratch (16-byte aligned)
    auto tsrc_bytes = [&](uint32_t i) -> uint64_t { return (out_px(i) * DI[i].pxsz + 15) & ~15ull; };
    if (sel) {   // windows for the rectangles that are not made of whole tiles, and for every turned, resized or tensor entry
        uint64_t need = 0, tab = 0, tmp = 0, tsz = 0, bsz = 0;
        for (uint32_t i = 0; i < n; i++) {
            const bool rs = sel[i].rs;
            if (DI[i].mode == 7) { }
            else if (shared(i)) { if (share[i].n) need += share[i].cover.h * window_pitch(share[i].cover, DI[i].pxsz); }
            else if (!whole_tiles(sel[i]) || turned(ops, i) || rs || fmt) need += sel[i].cover.h * window_pitch(sel[i], DI[i].pxsz);
            if (rs) { tab += resize_tab_bytes(sel[i]); tmp += resize_tmp_bytes(sel[i], DI[i].pxsz); }
            if ((rs || staged(i)) && fmt) tsz += tsrc_bytes(i);
            if (blurred(i) || augmented(i)) bsz += tsrc_bytes(i);
        }
        if (need) ENSURE(region, need);
        if (tab) ENSURE(rtab, tab);
        if (tmp) ENSURE(rtmp, tmp);
        if (tsz) ENSURE(tsrc, tsz);
        if (bsz) ENSURE(bscr, bsz);
    }
    // resampled entry i: the span of its crop at src (rows `pitch` bytes apart) resampled, and its window written into out
    // through its op, each pass reading the previous one's packed rows
    uint64_t tpos = 0, mpos = 0;
    auto resize_desc = [&](uint32_t i, uint64_t src, uint64_t pitch, uint8_t* out, uint32_t op) -> int {
        const RegionSel& R = sel[i];
        const xpngb_rect &r = R.rect, &c = R.crop, &win = R.win;
        ResizeDesc d{};
        d.coef = (uint64_t)ctx->rtab.p + tpos; tpos += resize_tab_bytes(R);
        const uint64_t tmp = (uint64_t)ctx->rtmp.p + mpos; mpos += resize_tmp_bytes(R, DI[i].pxsz);
        d.in_w = (uint32_t)c.w; d.in_h = (uint32_t)c.h; d.out_w = (uint32_t)win.w; d.out_h = (uint32_t)win.h;
        d.full_w = R.full.w; d.full_h = R.full.h; d.wx = (uint32_t)win.x; d.wy = (uint32_t)win.y;
        d.bx = (uint32_t)(r.x - c.x); d.by = (uint32_t)(r.y - c.y);
        d.filter = R.filter; d.pxsz = DI[i].pxsz; d.op = op;
        d.kx = resize_kx(R); d.ky = resize_ky(R);
        if (!d.kx) d.v = ResizePass{ src, pitch, (uint64_t)out, d.out_w, 1 };
        else if (!d.ky) d.h = ResizePass{ src, pitch, (uint64_t)out, d.out_h, 1 };
        else if (resize_vfirst(c.w, c.h, R.full.w, R.full.h)) {
            d.v = ResizePass{ src, pitch, tmp, (uint32_t)r.w, 0 };
            d.h = ResizePass{ tmp, r.w * DI[i].pxsz, (uint64_t)out, d.out_h, 1 };
        } else {
            d.h = ResizePass{ src, pitch, tmp, (uint32_t)r.h, 0 };
            d.v = ResizePass{ tmp, (uint64_t)d.out_w * DI[i].pxsz, (uint64_t)out, d.out_w, 1 };
        }
        d.first_coef = (uint32_t)rcoef; d.first_h = (uint32_t)rh; d.first_v = (uint32_t)rv;
        d.h_tiles_x = (d.out_w + RH_X - 1) / RH_X;
        rcoef += (d.kx ? d.out_w : 0) + (d.ky ? d.out_h : 0);
        if (d.kx) rh += (uint64_t)d.h_tiles_x * ((d.h.n + RH_ROWS - 1) / RH_ROWS);
        if (d.ky) rv += ((uint64_t)d.v.n * d.pxsz + RV_X - 1) / RV_X * ((d.out_h + RV_ROWS - 1) / RV_ROWS);
        if (rcoef > 0xFFFFFFFFull || rh > 0x7FFFFFFFull || rv > 0x7FFFFFFFull) FAIL("too many pixels for one resize launch");
        rdescs.push_back(d);
        return 0;
    };
    // tensor entry i: its w x h pixels at src (rows `pitch` bytes apart) written as its tensor at out through its op
    auto tensor_desc = [&](uint32_t i, uint64_t src, uint64_t pitch, uint64_t w, uint64_t h, uint8_t* out) -> int {
        TensorDesc d{};
        d.src = src; d.src_pitch = pitch; d.dst = (uint64_t)out; d.w = (uint32_t)w; d.h = (uint32_t)h;
        d.pxsz = DI[i].pxsz; d.c = fmt->channels == 3 ? 3 : DI[i].pxsz; d.op = ops ? (uint32_t)ops[i] : (uint32_t)OP_TL;
        d.tiles_x = (d.w + TT - 1) / TT; d.first_cta = (uint32_t)tctas;
        tctas += (uint64_t)d.tiles_x * ((d.h + TT - 1) / TT);
        if (tctas > 0x7FFFFFFFull) FAIL("too many pixels for one tensor launch");
        tdescs.push_back(d);
        return 0;
    };
    // coloured entry i: its npx packed pixels at px, changed in place
    auto color_desc = [&](uint32_t i, uint8_t* px, uint64_t npx) -> int {
        const xpngb_color& c = colors[i];
        ColorDesc d{};
        d.px = (uint64_t)px; d.npx = npx; d.pxsz = DI[i].pxsz; d.on = c.on; d.gray = c.gray;
        for (int k = 0; k < 3; k++) d.fac[k] = (float)c.factor[k];   // Pillow's ImagingBlend takes the factor as a float
        d.hue = (uint8_t)(int32_t)(c.factor[XPNGB_CJ_HUE] * 255.0);   // np.array(h * 255).astype(np.uint8): truncate, then wrap
        d.pre = 4;
        for (uint32_t s = 0; s < 4; s++) { d.order[s] = c.order[s]; if (c.order[s] == XPNGB_CJ_CONTRAST) d.pre = s; }
        d.first_cta = (uint32_t)cctas; d.mfirst_cta = (uint32_t)mctas;
        const uint64_t ctas = (npx + CL_PX - 1) / CL_PX;
        cctas += ctas;
        if ((c.on >> XPNGB_CJ_CONTRAST) & 1) mctas += ctas;
        if (cctas > 0x7FFFFFFFull) FAIL("too many pixels for one colour launch");
        cdescs.push_back(d);
        return 0;
    };
    // blurred entry i: its w x h packed pixels at px go through its passes, ping-ponged with its scratch; *res is where the
    // last pass leaves them.  swap: the entry is staged un-turned and k_to_tensor turns it a quarter, so the passes of the
    // output's x axis run along the staged columns, first.
    auto blur_desc = [&](uint32_t i, uint8_t* px, uint8_t* scr, uint64_t w, uint64_t h, bool swap, uint8_t** res) -> int {
        const xpngb_blur& b = blurs[i];
        const uint32_t pxsz = DI[i].pxsz;
        uint8_t* const buf[2] = { px, scr };
        uint32_t k = 0;
        auto pass = [&](uint32_t vert, const BlurBox& bx) {
            BlurPass& p = bstage[k].emplace_back();
            p.src = (uint64_t)buf[k & 1]; p.dst = (uint64_t)buf[(k + 1) & 1]; p.pitch = w * pxsz;
            p.w = (uint32_t)w; p.h = (uint32_t)h; p.pxsz = pxsz; p.vert = vert;
            p.ri = (uint32_t)bx.ri; p.ww = bx.ww; p.fw = bx.fw; p.t = 256;
            k++;
        };
        for (uint32_t a = 0; a < 2; a++) {   // output x, then output y
            const float r = (float)b.radius[a];
            if (r == 0.f) continue;
            const BlurBox bx = blur_box(r);
            for (int rep = 0; rep < 3; rep++) pass(a == 0 ? (swap ? 1u : 0u) : (swap ? 0u : 1u), bx);
        }
        const BlurBox id{ 0, 1u << 24, 0 };   // the identity pass: out = (p * 2^24 + 2^23) >> 24 = p
        if (k == 0) pass(1, id);               // solarize alone
        if (!fmt && (k & 1)) pass(1, id);      // a uint8 entry's result belongs at its output
        if (b.solarize) bstage[k - 1].back().t = solarize_t(b.threshold);
        *res = buf[k & 1];
        return 0;
    };
    // augmented entry i: its w x h staged pixels at px, turned by eop into the output image, go through its program; the
    // warps and SHARPNESS ping-pong with its scratch scr, and *res is where the last step leaves the pixels (px for a uint8
    // entry, whose eop is OP_TL: its pixels are staged as written)
    auto aug_desc = [&](uint32_t i, uint8_t* px, uint8_t* scr, uint64_t w, uint64_t h, uint32_t eop, uint8_t** res) -> int {
        const xpngb_augment& A = augs[i];
        const uint32_t pxsz = DI[i].pxsz;
        const uint64_t npx = w * h;
        const bool q = eop == OP_R90 || eop == OP_R270;
        const double W = (double)(q ? h : w), H = (double)(q ? w : h);
        uint8_t *cur = px, *other = scr;
        auto pix = [&](uint32_t k, uint32_t mode) -> AugPix& {
            AugPix& d = apix[k].emplace_back();
            d.src = (uint64_t)cur; d.dst = (uint64_t)other; d.w = (uint32_t)w; d.h = (uint32_t)h; d.pxsz = pxsz; d.eop = eop; d.mode = mode;
            d.first_cta = (uint32_t)apctas[k];
            apctas[k] += (npx + AP_THREADS - 1) / AP_THREADS;
            uint8_t* t = cur; cur = other; other = t;
            return d;
        };
        for (uint32_t k = 0; k < A.nsteps; k++) {
            const xpngb_aug_step& s = A.step[k];
            const double* a = s.data;
            if (s.kind == XPNGB_AUG_AFFINE) {
                const uint32_t mode = s.arg == 2 ? AP_BILINEAR : s.arg == 3 ? AP_BICUBIC
                                      : a[1] != 0.0 || a[3] != 0.0 ? (affine_fixed_ok(a, W, H) ? AP_FIXED : AP_SEQ) : AP_SEQ;
                AugPix& d = pix(k, mode);
                memcpy(d.fill, s.fill, 4);
                if (mode == AP_FIXED) {
                    const double v[6] = { a[0], a[1], a[2] + a[0] * 0.5 + a[1] * 0.5, a[3], a[4], a[5] + a[3] * 0.5 + a[4] * 0.5 };
                    for (int c = 0; c < 6; c++) d.fx[c] = pil_fix(v[c]);
                } else if (mode == AP_SEQ && a[1] == 0.0 && a[3] == 0.0) {   // ImagingScaleAffine: x per column, y per row
                    const double v[6] = { a[2] + a[0] * 0.5, 0.0, a[0], a[5] + a[4] * 0.5, a[4], 0.0 };
                    memcpy(d.a, v, sizeof v);
                } else if (mode == AP_SEQ) {   // ImagingTransformAffine's double path
                    const double v[6] = { a[2] + a[1] * 0.5 + a[0] * 0.5, a[1], a[0], a[5] + a[4] * 0.5 + a[3] * 0.5, a[4], a[3] };
                    memcpy(d.a, v, sizeof v);
                } else memcpy(d.a, a, sizeof d.a);
            } else if (s.kind == XPNGB_AUG_TRANSPOSE) {
                pix(k, AP_TRANSPOSE).top = (uint32_t)s.arg;
            } else if (s.kind == XPNGB_AUG_SHARPNESS) {
                pix(k, AP_SHARP).fac = (float)s.value;
            } else if (s.kind == XPNGB_AUG_BRIGHTNESS || s.kind == XPNGB_AUG_COLOR || s.kind == XPNGB_AUG_CONTRAST) {
                const uint32_t step = s.kind == XPNGB_AUG_BRIGHTNESS ? XPNGB_CJ_BRIGHTNESS : s.kind == XPNGB_AUG_COLOR ? XPNGB_CJ_SATURATION
                                                                                                                    : XPNGB_CJ_CONTRAST;
                ColorDesc d{};   // colour decode with this one step on
                d.px = (uint64_t)cur; d.npx = npx; d.pxsz = pxsz; d.on = 1u << step;
                d.fac[step] = (float)s.value;
                for (uint32_t c = 0; c < 4; c++) d.order[c] = (uint8_t)c;
                d.pre = XPNGB_CJ_CONTRAST;
                d.first_cta = (uint32_t)acctas[k]; d.mfirst_cta = (uint32_t)amctas[k];
                const uint64_t ctas = (npx + CL_PX - 1) / CL_PX;
                acctas[k] += ctas;
                if (step == XPNGB_CJ_CONTRAST) amctas[k] += ctas;
                acol[k].push_back(d);
            } else {
                AugLut& d = alut[k].emplace_back();
                d.px = (uint64_t)cur; d.npx = npx; d.pxsz = pxsz; d.kind = s.kind; d.hist = 0;
                d.first_cta = (uint32_t)alctas[k]; d.hfirst_cta = (uint32_t)ahctas[k];
                alctas[k] += (npx + CL_PX - 1) / CL_PX;
                const uint32_t t = solarize_t(s.value), keep = s.kind == XPNGB_AUG_POSTERIZE ? ~((1u << (8 - s.arg)) - 1) : 255u;
                for (uint32_t v = 0; v < 256; v++) {
                    const uint32_t o = s.kind == XPNGB_AUG_POSTERIZE ? v & keep : s.kind == XPNGB_AUG_SOLARIZE ? (v < t ? v : 255 - v) : 255 - v;
                    d.lut[v] = d.lut[256 + v] = d.lut[512 + v] = (uint8_t)o;
                }
                if (s.kind == XPNGB_AUG_EQUALIZE || s.kind == XPNGB_AUG_AUTOCONTRAST) {   // from the histograms, on the device
                    d.hist = 1 + anhist[k]++;   // the histogram's number + 1 until the layout is known
                    ahctas[k] += (npx + AH_PX - 1) / AH_PX;
                }
            }
            if (apctas[k] > 0x7FFFFFFFull || acctas[k] > 0x7FFFFFFFull || alctas[k] > 0x7FFFFFFFull) FAIL("too many pixels for one augment launch");
        }
        if (!fmt && cur != px) pix(A.nsteps, AP_TRANSPOSE).top = OP_TL;   // a uint8 entry's result belongs at its output
        *res = cur;
        return 0;
    };
    // entry i of a region call: its rectangle at src (rows `pitch` bytes apart) cropped, turned, resized or made a tensor
    uint64_t spos = 0, bpos = 0;
    auto region_out = [&](uint32_t i, uint64_t src, uint64_t pitch, uint8_t* out) -> int {
        const xpngb_rect& r = sel[i].rect;
        const uint32_t pxsz = DI[i].pxsz;
        if (fmt && (sel[i].rs || staged(i))) {   // uint8 pixels in tsrc, resampled or copied without the op; k_to_tensor applies it
            uint8_t* t = (uint8_t*)ctx->tsrc.p + spos;
            spos += tsrc_bytes(i);
            const uint64_t w = sel[i].rs ? sel[i].win.w : r.w, h = sel[i].rs ? sel[i].win.h : r.h;
            if (sel[i].rs) { if (resize_desc(i, src, pitch, t, OP_TL)) return 1; }
            else crops.push_back(CropDesc{ src, (uint64_t)t, pitch, (uint32_t)(r.w * pxsz), (uint32_t)r.h });
            uint8_t* scr = nullptr;
            if (blurred(i) || augmented(i)) { scr = (uint8_t*)ctx->bscr.p + bpos; bpos += tsrc_bytes(i); }
            if (augmented(i)) {   // the blur then ping-pongs between the buffer the program ended in and the other one
                uint8_t* r;
                if (aug_desc(i, t, scr, w, h, ops ? (uint32_t)ops[i] : (uint32_t)OP_TL, &r)) return 1;
                if (r != t) { scr = t; t = r; }
            }
            if (colored(i) && color_desc(i, t, w * h)) return 1;
            if (blurred(i) && blur_desc(i, t, scr, w, h, quarter(ops, i), &t)) return 1;
            return tensor_desc(i, (uint64_t)t, w * pxsz, w, h, out);
        }
        if (fmt) return tensor_desc(i, src, pitch, r.w, r.h, out);
        if (sel[i].rs) return resize_desc(i, src, pitch, out, ops ? (uint32_t)ops[i] : (uint32_t)OP_TL);
        if (!turned(ops, i)) crops.push_back(CropDesc{ src, (uint64_t)out, pitch, (uint32_t)(r.w * pxsz), (uint32_t)r.h });
        else if (!orient_desc(odescs.emplace_back(), src, pitch, (uint64_t)out, r.w, r.h, pxsz, ops[i], &octas))
            FAIL("too many pixels for one orientation launch");
        return 0;
    };
    uint64_t wpos = 0, gwin = 0, gpitch = 0;   // the window of the current group of a shared file, and its cover
    xpngb_rect gcov{};
    for (uint32_t i = 0; i < n; i++) {
        DecImage& D = DI[i];
        uint8_t* out = dpx + imgs[i].offset;
        const int sfac = any2 ? 4 : 1;
        if (!sel) {
            const TileGrid g = tile_grid(D.w, D.h);
            plan_image(P, g, all_tiles(g), (uint64_t)out, (uint64_t)D.w * D.pxsz, 0, 0, D.w, D.h, D.pxsz, D.mode, sfac, 0);
            D.gcols = (uint32_t)g.nw; D.r0 = 0; D.c0 = 0; D.nrows = (uint32_t)g.nh; D.ncols = (uint32_t)g.nw;
        } else if (D.mode == 7) {   // no tiles: the rectangle's rows are read from the file
            const xpngb_rect& r = sel[i].rect;
            ImageDesc I{}; I.tile0 = (uint32_t)P.tiles.size(); I.mode = 7; I.w = D.w; I.h = D.h; I.pxsz = D.pxsz;
            P.imgs.push_back(I);
            const uint64_t src = (uint64_t)(din + D.file_off + 8 + (r.y * D.w + r.x) * D.pxsz);   // any byte alignment
            if (region_out(i, src, (uint64_t)D.w * D.pxsz, out)) return 1;
        } else if (shared(i)) {   // never in place: the window holds every entry of the group
            const RegionSel& R = sel[i];
            const xpngb_rect& r = R.rect;
            if (share[i].n) {
                gcov = share[i].cover; gpitch = window_pitch(gcov, D.pxsz); gwin = (uint64_t)ctx->region.p + wpos;
                const TileSel& s = share[i].s;
                plan_image(P, R.g, s, gwin, gpitch, gcov.x, gcov.y, D.w, D.h, D.pxsz, D.mode, sfac, 0);
                wpos += gcov.h * gpitch;
                D.r0 = (uint32_t)s.r0; D.c0 = (uint32_t)s.c0; D.nrows = (uint32_t)(s.r1 - s.r0 + 1); D.ncols = (uint32_t)(s.c1 - s.c0 + 1);
            } else {   // no tiles of its own: k_dec_tile_offsets walks no row of it
                ImageDesc I{}; I.tile0 = (uint32_t)P.tiles.size(); I.mode = D.mode; I.w = D.w; I.h = D.h; I.pxsz = D.pxsz;
                P.imgs.push_back(I);
                D.r0 = 0; D.c0 = 0; D.nrows = 0; D.ncols = 0;
            }
            D.gcols = (uint32_t)R.g.nw;
            if (region_out(i, gwin + (r.y - gcov.y) * gpitch + (r.x - gcov.x) * D.pxsz, gpitch, out)) return 1;
        } else {
            const RegionSel& R = sel[i];
            const xpngb_rect &r = R.rect, &c = R.cover;
            if (whole_tiles(R) && !turned(ops, i) && !R.rs && !fmt)
                plan_image(P, R.g, R.s, (uint64_t)out, r.w * D.pxsz, r.x, r.y, D.w, D.h, D.pxsz, D.mode, sfac, 0);
            else {   // a turned, resized or tensor rectangle cannot be decoded in place, even when it is made of whole tiles
                const uint64_t pitch = window_pitch(R, D.pxsz), win = (uint64_t)ctx->region.p + wpos;
                plan_image(P, R.g, R.s, win, pitch, c.x, c.y, D.w, D.h, D.pxsz, D.mode, sfac, 0);
                if (region_out(i, win + (r.y - c.y) * pitch + (r.x - c.x) * D.pxsz, pitch, out)) return 1;
                wpos += c.h * pitch;
            }
            D.gcols = (uint32_t)R.g.nw; D.r0 = (uint32_t)R.s.r0; D.c0 = (uint32_t)R.s.c0;
            D.nrows = (uint32_t)(R.s.r1 - R.s.r0 + 1); D.ncols = (uint32_t)(R.s.c1 - R.s.c0 + 1);
        }
        D.tile0 = P.imgs[i].tile0; D.ntiles = P.imgs[i].ntiles;
        if (!fmt && (augmented(i) || colored(i) || blurred(i))) {   // uint8 output: changed where it is written, as written
            uint64_t w = sel[i].rs ? sel[i].win.w : sel[i].rect.w, h = sel[i].rs ? sel[i].win.h : sel[i].rect.h;
            if (quarter(ops, i)) { const uint64_t t = w; w = h; h = t; }
            uint8_t *scr = nullptr, *res;
            if (blurred(i) || augmented(i)) { scr = (uint8_t*)ctx->bscr.p + bpos; bpos += tsrc_bytes(i); }
            if (augmented(i) && aug_desc(i, out, scr, w, h, OP_TL, &res)) return 1;
            if (colored(i) && color_desc(i, out, out_px(i))) return 1;
            if (blurred(i) && blur_desc(i, out, scr, w, h, false, &res)) return 1;
        }
    }
    // blur passes stage by stage, each stage's CTAs numbered from 0
    size_t bpasses = 0;
    uint32_t nstage = 0;
    uint64_t bctas[BLUR_STAGES] = {};
    for (uint32_t k = 0; k < BLUR_STAGES; k++) {
        for (BlurPass& p : bstage[k]) {
            p.first_cta = (uint32_t)bctas[k];
            bctas[k] += ((uint64_t)(p.vert ? p.w : p.h) * p.pxsz + BL_THREADS - 1) / BL_THREADS;
            if (bctas[k] > 0x7FFFFFFFull) FAIL("too many pixels for one blur launch");
        }
        bpasses += bstage[k].size();
        if (!bstage[k].empty()) nstage = k + 1;
    }
    // augment stages in the lane's adescs: first every stage's AugPix, ColorDesc and AugLut (uploaded), then every stage's
    // luma sums and histograms (zeroed)
    struct AugAt { size_t pix, col, lut, sum, hist; };
    AugAt aat[AUG_STAGES] = {};
    size_t adesc_bytes = 0, azero_bytes = 0;
    uint32_t anstage = 0;
    for (uint32_t k = 0; k < AUG_STAGES; k++) {
        aat[k].pix = adesc_bytes; adesc_bytes += apix[k].size() * sizeof(AugPix);
        aat[k].col = adesc_bytes; adesc_bytes += acol[k].size() * sizeof(ColorDesc);
        aat[k].lut = adesc_bytes; adesc_bytes += alut[k].size() * sizeof(AugLut);
        aat[k].sum = azero_bytes; azero_bytes += acol[k].size() * 8;
        aat[k].hist = azero_bytes; azero_bytes += (size_t)anhist[k] * 3 * 256 * 8;
        if (!apix[k].empty() || !acol[k].empty() || !alut[k].empty()) anstage = k + 1;
    }
    adesc_bytes = (adesc_bytes + 15) & ~(size_t)15;
    if (anstage) {
        ENSURE(adescs, adesc_bytes + azero_bytes);
        uint8_t* zero = (uint8_t*)ctx->adescs.p + adesc_bytes;
        for (uint32_t k = 0; k < anstage; k++)
            for (AugLut& d : alut[k]) if (d.hist) d.hist = (uint64_t)(zero + aat[k].hist + (d.hist - 1) * 3 * 256 * 8);
    }
    if (P.tiles.size() > (1u << 24) || P.seg_tile.size() > (1u << 28)) FAIL("too many tiles for one chunk (%zu)", P.tiles.size());
    const uint32_t ntiles = (uint32_t)P.tiles.size();
    ctx->root->decoded_tiles += ntiles;
    if (upload_plan(ctx, P)) return 1;
    ENSURE(dimgs, n * sizeof(DecImage)); ENSURE(dtiles, ntiles * sizeof(DecTile)); ENSURE(errflag, 4);
    // pinned staging: DecImage table, stored-file starts, error flag (64 bytes), crop, orientation, resize and tensor descriptors
    const size_t pin_crops = n * (sizeof(DecImage) + 8) + 64, pin_orients = pin_crops + crops.size() * sizeof(CropDesc);
    const size_t pin_resize = pin_orients + odescs.size() * sizeof(OrientDesc), pin_tensor = pin_resize + rdescs.size() * sizeof(ResizeDesc);
    const size_t pin_color = pin_tensor + tdescs.size() * sizeof(TensorDesc), pin_blur = pin_color + cdescs.size() * sizeof(ColorDesc);
    const size_t pin_aug = pin_blur + bpasses * sizeof(BlurPass);
    if (ensure_pin(ctx, ctx->pin_b, pin_aug + (anstage ? adesc_bytes : 0))) return 1;
    memcpy(ctx->pin_b.p, DI.data(), n * sizeof(DecImage));
    CK(cudaMemcpyAsync(ctx->dimgs.p, ctx->pin_b.p, n * sizeof(DecImage), cudaMemcpyHostToDevice, ctx->stream));
    if (any7 && !sel) {   // where each stored image's file starts (k_load7), ~0 = not a stored image
        uint64_t* cf = (uint64_t*)((uint8_t*)ctx->pin_b.p + n * sizeof(DecImage));
        for (uint32_t i = 0; i < n; i++) cf[i] = DI[i].mode == 7 ? DI[i].file_off : ~0ull;
        ENSURE(offs, n * 8);
        CK(cudaMemcpyAsync(ctx->offs.p, cf, n * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!crops.empty()) {
        ENSURE(crops, crops.size() * sizeof(CropDesc));
        memcpy((uint8_t*)ctx->pin_b.p + pin_crops, crops.data(), crops.size() * sizeof(CropDesc));
        CK(cudaMemcpyAsync(ctx->crops.p, (uint8_t*)ctx->pin_b.p + pin_crops, crops.size() * sizeof(CropDesc), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!odescs.empty()) {   // this lane's staging and descriptor buffer: the lanes of a call run concurrently
        const size_t nb = odescs.size() * sizeof(OrientDesc);
        ENSURE(orients, nb);
        memcpy((uint8_t*)ctx->pin_b.p + pin_orients, odescs.data(), nb);
        CK(cudaMemcpyAsync(ctx->orients.p, (uint8_t*)ctx->pin_b.p + pin_orients, nb, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!rdescs.empty()) {
        const size_t nb = rdescs.size() * sizeof(ResizeDesc);
        ENSURE(rdescs, nb);
        memcpy((uint8_t*)ctx->pin_b.p + pin_resize, rdescs.data(), nb);
        CK(cudaMemcpyAsync(ctx->rdescs.p, (uint8_t*)ctx->pin_b.p + pin_resize, nb, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (!tdescs.empty()) {
        const size_t nb = tdescs.size() * sizeof(TensorDesc);
        ENSURE(tdescs, nb);
        memcpy((uint8_t*)ctx->pin_b.p + pin_tensor, tdescs.data(), nb);
        CK(cudaMemcpyAsync(ctx->tdescs.p, (uint8_t*)ctx->pin_b.p + pin_tensor, nb, cudaMemcpyHostToDevice, ctx->stream));
    }
    const size_t csum = cdescs.size() * sizeof(ColorDesc);   // the luma sums follow the descriptors (8-byte aligned)
    if (!cdescs.empty()) {
        ENSURE(cdescs, csum + cdescs.size() * 8);
        memcpy((uint8_t*)ctx->pin_b.p + pin_color, cdescs.data(), csum);
        CK(cudaMemcpyAsync(ctx->cdescs.p, (uint8_t*)ctx->pin_b.p + pin_color, csum, cudaMemcpyHostToDevice, ctx->stream));
        if (mctas) CK(cudaMemsetAsync((uint8_t*)ctx->cdescs.p + csum, 0, cdescs.size() * 8, ctx->stream));
    }
    if (bpasses) {
        ENSURE(bdescs, bpasses * sizeof(BlurPass));
        size_t at = pin_blur;
        for (uint32_t k = 0; k < nstage; k++) {
            memcpy((uint8_t*)ctx->pin_b.p + at, bstage[k].data(), bstage[k].size() * sizeof(BlurPass));
            at += bstage[k].size() * sizeof(BlurPass);
        }
        CK(cudaMemcpyAsync(ctx->bdescs.p, (uint8_t*)ctx->pin_b.p + pin_blur, bpasses * sizeof(BlurPass), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (anstage) {
        uint8_t* pa = (uint8_t*)ctx->pin_b.p + pin_aug;
        for (uint32_t k = 0; k < anstage; k++) {
            memcpy(pa + aat[k].pix, apix[k].data(), apix[k].size() * sizeof(AugPix));
            memcpy(pa + aat[k].col, acol[k].data(), acol[k].size() * sizeof(ColorDesc));
            memcpy(pa + aat[k].lut, alut[k].data(), alut[k].size() * sizeof(AugLut));
        }
        CK(cudaMemcpyAsync(ctx->adescs.p, pa, adesc_bytes, cudaMemcpyHostToDevice, ctx->stream));
        if (azero_bytes) CK(cudaMemsetAsync((uint8_t*)ctx->adescs.p + adesc_bytes, 0, azero_bytes, ctx->stream));
    }
    CK(cudaMemsetAsync(ctx->errflag.p, 0, 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->dtiles.p, 0, ntiles * sizeof(DecTile), ctx->stream));
    const TileDesc* d_tiles = (const TileDesc*)ctx->tiles.p;
    const DecImage* d_imgs = (const DecImage*)ctx->dimgs.p;
    DecTile* d_dt = (DecTile*)ctx->dtiles.p;
    int* d_err = (int*)ctx->errflag.p;
    const uint32_t nseg = (uint32_t)P.seg_tile.size();
    const uint32_t* d_seg_tile = (const uint32_t*)ctx->seg_tile.p;
    bool side_busy[xpngb_ctx::NSIDE] = {};
    const uint32_t pd_cap = 17u * ntiles;
    if (any1 || any2) {
        ENSURE(streams, P.str_total); ENSURE(nlseq, P.px_total); ENSURE(rows, P.row_total * sizeof(RowInfo));
        ENSURE(rowcnt, P.row_total * 4); ENSURE(edge, P.row_total * 16);
        ENSURE(ccnt, (size_t)nseg * 9 * 4); ENSURE(cbit, (size_t)nseg * 4); ENSURE(resv, (P.px_total + 4 * P.row_total) * 4);
        if (P.any_rgba) { ENSURE(alpha, P.px_total); ENSURE(plane, P.px_total); }
        if (!lat) { ENSURE(pdw, 2 * pdw_bytes(pd_cap)); CK(cudaMemsetAsync(ctx->pdw.p, 0, 2 * pdw_bytes(pd_cap), ctx->stream)); }
        LAUNCH_HI(k_dec_tile_offsets, (n + 127) / 128, 128, 0, d_imgs, din, d_dt, n, d_err);
    }
    // Stream plan of one chunk.  Main stream: the level-2 family (or the only family).  side[2]: the level-1 family
    // when both are present (config 0: the corpus mixes RGB and RGBA files).  side[0], side[1]: level-2
    // value streams.  side[3]: the alpha plane.  Each family's chain is parse -> context rANS -> context walk.
    uint32_t maxpx = 0;
    for (const TileDesc& t : P.tiles) if (t.npx > maxpx) maxpx = t.npx;
    const uint32_t wsm = (maxpx / 8 + 32) * 4;          // nibble-packed streams of the largest tile + pad words
    PdWork Wl[3] = {};                              // work lists of the pair decoders / the batch walk, per level family
    auto launch_walk = [&](uint32_t mode) -> int {
        WalkArgs wa{ d_tiles, d_imgs, d_dt, (const uint8_t*)ctx->streams.p, (uint8_t*)ctx->nlseq.p, ntiles, mode };
        if (!lat && !ctx->root->walk_ring) {   // batches: three tiles per warp, longest tiles first
            const PdWork& W = Wl[mode];
            LAUNCH_HI(k_dec_walk3<2>, (ntiles + 5) / 6, 64, 0, wa, (const uint32_t*)(W.order + (size_t)PD_WALK * W.cap), (const uint32_t*)(W.total + PD_WALK));
            return 0;
        }
        // the shared-memory walk only pays when every tile's CTA of the CALL is resident at once (no waves): 227 KB per SM, 148 SMs
        const uint32_t resident = 148u * ((227u * 1024u) / (wsm + 1024u));
        if (call_tiles <= resident && maxpx <= WALK_SMEM_MAX_SYMS && !ctx->root->walk_ring) LAUNCH_HI(k_dec_walk_smem<0>, ntiles, 32, wsm, wa);
        else if (call_tiles <= 592) LAUNCH_HI(k_dec_walk_ring<1>, ntiles, 32, 0, wa);
        else LAUNCH_HI(k_dec_walk_ring<4>, (ntiles + 3) / 4, 128, 0, wa);
        return 0;
    };
    // pair decoders of one level family: work lists, run / raw fills, then one launch per class
    auto pd_lists = [&](uint32_t mode, PdWork& W) -> int {
        W = pdw_at((uint8_t*)ctx->pdw.p + (mode == 1 ? 0 : pdw_bytes(pd_cap)), pd_cap);
        const unsigned g = (17u * ntiles + 255) / 256;
        LAUNCH_HI(k_pd_count, g, 256, 0, d_tiles, d_imgs, (const DecTile*)d_dt, ntiles, mode, W);
        LAUNCH_HI(k_pd_scan, PD_NCLASS, 1024, 0, W);
        LAUNCH_HI(k_pd_fill, g, 256, 0, d_tiles, d_imgs, (const DecTile*)d_dt, ntiles, mode, W);
        return 0;
    };
    auto pd_args = [&](const PdWork& W, int cls) {
        return PairDecArgs{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, (uint8_t*)ctx->alpha.p, W.order + (size_t)cls * W.cap, W.total + cls, d_err };
    };
    auto pd_grid = [&](uint32_t per_tile) { return (unsigned)(((uint64_t)per_tile * ntiles + PD_BLK * PD_WARPS - 1) / (PD_BLK * PD_WARPS)); };
    if (any1) {
        const bool own_stream = any2;                   // level-1 family next to a level-2 family
        cudaStream_t f1 = own_stream ? side_of(ctx, 2) : ctx->stream;
        if (own_stream) { FORK_SIDE(2); side_busy[2] = true; }
        LAUNCH_HI(k_dec_parse_m1, (ntiles + 127) / 128, 128, 0, d_tiles, d_imgs, din, d_dt, ntiles, d_err);
        RansDecArgs ra{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, (uint8_t*)ctx->alpha.p, ntiles, 0, 9, d_err };
        AlphaArgs al{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->alpha.p, (uint8_t*)ctx->plane.p, (uint32_t*)ctx->rowcnt.p };
        if (lat) {
            if (P.any_rgba) {                             // the alpha plane is independent of the context walk
                FORK_FROM(f1, 3); side_busy[3] = true;
                RansDecArgs rb = ra; rb.c0 = 9; rb.nc = 1;
                auto k_dec_rans_v2_lat_alpha = k_dec_rans_v2_lat;
                LAUNCH_HI(k_dec_rans_v2_lat_alpha, ntiles, 32, lat_smem(LUT_TWO_15), rb, LUT_TWO_15);
                LAUNCH(k_dec_alpha, ntiles, 256, 0, al);
                LAUNCH(k_dec_rows_rgba, ntiles, 32, 0, d_tiles, d_imgs, (const DecTile*)d_dt, (const uint32_t*)ctx->rowcnt.p, (RowInfo*)ctx->rows.p);
            }
            ctx->cur = f1;
            auto k_dec_rans_v2_lat_two = k_dec_rans_v2_lat;   // the two-level table's name in the profile report
            if (call_tiles <= ctx->root->v2_direct_max_tiles) LAUNCH_HI(k_dec_rans_v2_lat, 9 * ntiles, 32, lat_smem(LUT_ONE_12), ra, LUT_ONE_12);
            else LAUNCH_HI(k_dec_rans_v2_lat_two, 9 * ntiles, 32, lat_smem(LUT_TWO_12), ra, LUT_TWO_12);
        } else {
            PdWork& W = Wl[1];
            if (pd_lists(1, W)) return 1;
            PdFillArgs fa{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, (uint8_t*)ctx->alpha.p, ntiles, 1 };
            LAUNCH_HI(k_pd_fill_blocks, (17u * ntiles + 3) / 4, 128, 0, fa);
            if (P.any_rgba) {
                FORK_FROM(f1, 3); side_busy[3] = true;
                auto k_dec_rans_pair_v2_alpha = k_dec_rans_pair<2, 0>;
                LAUNCH_HI(k_dec_rans_pair_v2_alpha, pd_grid(1), PD_WARPS * 32, PD_WARPS * PD_BIG_BYTES, pd_args(W, PD_BIG));
                LAUNCH(k_dec_alpha, ntiles, 256, 0, al);
                LAUNCH(k_dec_rows_rgba, ntiles, 32, 0, d_tiles, d_imgs, (const DecTile*)d_dt, (const uint32_t*)ctx->rowcnt.p, (RowInfo*)ctx->rows.p);
            }
            ctx->cur = f1;
            auto k_dec_rans_pair_v2_ctx = k_dec_rans_pair<2, 8>;
            LAUNCH_HI(k_dec_rans_pair_v2_ctx, pd_grid(9), PD_WARPS * 32, 0, pd_args(W, PD_S8));
        }
        if (launch_walk(1)) return 1;
        BACK_TO_MAIN();
    }
    if (any2) {
        LAUNCH_HI(k_dec_parse_m2, (ntiles + 127) / 128, 128, 0, d_tiles, d_imgs, din, d_dt, ntiles, d_err);
        if (lat) {
            // value streams on the side streams (joined before the residual kernels); LAT_M2_ORDER: 0..2 alphabets of at
            // most 16 symbols (direct table, 64 KiB), 3..7 larger alphabets (two-level), 8..16 contexts, 17 grey plane
            // a batch with more chains than fit next to 64 KiB tables (3 per SM) trades the shorter dependent step of the
            // direct table for residency: two-level tables (17 KiB) keep 12 chains per SM
            const bool direct = call_tiles <= ctx->root->direct_max_tiles;
            const uint32_t lut16 = direct ? LUT_ONE_14 : LUT_TWO_14;
            RansV1LatArgs la{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, ntiles, 0, 3, lut16, 0u, ~0u, d_err };
            auto k_dec_rans_v1_lat_values16 = k_dec_rans_v1_lat; auto k_dec_rans_v1_lat_values256 = k_dec_rans_v1_lat;
            auto k_dec_rans_v1_lat_grey = k_dec_rans_v1_lat; auto k_dec_rans_v1_lat_ctx = k_dec_rans_v1_lat;   // names for the profile report
            auto k_dec_rans_v1_lat_ctx_short = k_dec_rans_v1_lat; auto k_dec_rans_v1_lat_values16_two = k_dec_rans_v1_lat;
            FORK_SIDE(0); side_busy[0] = true;
            if (direct) LAUNCH_HI(k_dec_rans_v1_lat_values16, 3 * ntiles, 32, lat_smem(lut16), la);
            else LAUNCH_HI(k_dec_rans_v1_lat_values16_two, 3 * ntiles, 32, lat_smem(lut16), la);
            FORK_SIDE(1); side_busy[1] = true;
            la.j0 = 3; la.nj = 5; la.lut_bytes = LUT_TWO_14;
            LAUNCH_HI(k_dec_rans_v1_lat_values256, 5 * ntiles, 32, lat_smem(LUT_TWO_14), la);
            la.j0 = 17; la.nj = 1; la.lut_bytes = LUT_TWO_15;
            LAUNCH_HI(k_dec_rans_v1_lat_grey, ntiles, 32, lat_smem(LUT_TWO_15), la);
            BACK_TO_MAIN();
            // context streams: the few long ones (they bound the walk's start on real images) get the 64 KiB direct table,
            // the many short ones a two-level table on a side stream, so that everything stays resident
            constexpr uint32_t CTX_LONG = 24576;
            la.j0 = 8; la.nj = 9; la.lut_bytes = LUT_TWO_14; la.n_lo = 0; la.n_hi = direct ? CTX_LONG : ~0u;
            if (direct) {
                FORK_SIDE(4); side_busy[4] = true;
                LAUNCH_HI(k_dec_rans_v1_lat_ctx_short, 9 * ntiles, 32, lat_smem(LUT_TWO_14), la);
                BACK_TO_MAIN();
                la.lut_bytes = LUT_ONE_14; la.n_lo = CTX_LONG; la.n_hi = ~0u;
                LAUNCH_HI(k_dec_rans_v1_lat_ctx, 9 * ntiles, 32, lat_smem(LUT_ONE_14), la);
                JOIN_SIDE(4); side_busy[4] = false;       // the walk needs every context stream
            } else LAUNCH_HI(k_dec_rans_v1_lat_ctx, 9 * ntiles, 32, lat_smem(LUT_TWO_14), la);
        } else {
            // the value streams (16-symbol alphabet: the longest chains of a tile; large alphabets) start first on the side
            // streams; contexts and the 8-symbol value streams on the main stream, followed by the walk
            PdWork& W = Wl[2];
            if (pd_lists(2, W)) return 1;
            PdFillArgs fa{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, (uint8_t*)ctx->alpha.p, ntiles, 2 };
            auto k_dec_rans_pair_v1_s16 = k_dec_rans_pair<1, 15>; auto k_dec_rans_pair_v1_big = k_dec_rans_pair<1, 0>; auto k_dec_rans_pair_v1_s8 = k_dec_rans_pair<1, 8>;
            FORK_SIDE(0); side_busy[0] = true;
            if (call_tiles <= ctx->root->s16_lat_max_tiles) {
                // few enough of the longest chains to be resident all at once as warp-per-block chains with a two-level table
                // (about 55 cycles per symbol, against about 170 per symbol and state of the pair decoder)
                RansV1LatArgs la{ d_tiles, d_imgs, d_dt, din, (uint8_t*)ctx->streams.p, ntiles, 0, 1, LUT_TWO_14, 0u, ~0u, d_err };
                auto k_dec_rans_v1_lat_st4 = k_dec_rans_v1_lat;
                LAUNCH_HI(k_dec_rans_v1_lat_st4, ntiles, 32, lat_smem(LUT_TWO_14), la);
            } else
            LAUNCH_HI(k_dec_rans_pair_v1_s16, pd_grid(1), PD_WARPS * 32, 0, pd_args(W, PD_S16));
            FORK_SIDE(1); side_busy[1] = true;
            LAUNCH_HI(k_dec_rans_pair_v1_big, pd_grid(5), PD_WARPS * 32, PD_WARPS * PD_BIG_BYTES, pd_args(W, PD_BIG));
            BACK_TO_MAIN();
            LAUNCH_HI(k_pd_fill_blocks, (17u * ntiles + 3) / 4, 128, 0, fa);   // run / raw blocks (contexts among them: before the walk)
            LAUNCH_HI(k_dec_rans_pair_v1_s8, pd_grid(11), PD_WARPS * 32, 0, pd_args(W, PD_S8));
        }
        if (launch_walk(2)) return 1;
    }
    // batches: RGB tiles with word-aligned rows get the row-pitched residual plane and k_dec_unpredict_rgb
    const uint32_t pitched = (!lat || call_tiles > ctx->root->unr_multi_max_tiles) ? 1u : 0u;
    bool all_pitched = true;
    for (const TileDesc& t : P.tiles) all_pitched &= tile_pitched(t);
    if (any1 || any2) {
        if (side_busy[2]) JOIN_SIDE(2);                   // the other family's nl sequences
        ChunkArgs ch{ d_tiles, d_seg_tile, d_imgs, d_dt, (const uint8_t*)ctx->nlseq.p, (const uint8_t*)ctx->streams.p, din,
                      (uint32_t*)ctx->ccnt.p, (uint32_t*)ctx->cbit.p, (uint32_t*)ctx->resv.p, ntiles, d_err, pitched };
        LAUNCH(k_dec_chunk_hist, nseg, 256, 0, ch);
        LAUNCH_HI(k_dec_chunk_scan, (ntiles + 3) / 4, 128, 0, ch);
        for (int k = 0; k < xpngb_ctx::NSIDE; k++) if (k != 2 && side_busy[k]) JOIN_SIDE(k);
        if (any1) LAUNCH(k_dec_residuals<1>, nseg, 256, 0, ch);
        if (any2) { LAUNCH(k_dec_residuals<2>, nseg, 256, 0, ch); LAUNCH(k_dec_residuals_grey, nseg, 256, 0, ch); }
        UnpredArgs ua{ d_tiles, d_imgs, d_dt, din, (const uint32_t*)ctx->resv.p, (const uint8_t*)ctx->plane.p, (const RowInfo*)ctx->rows.p,
                       (uint4*)ctx->edge.p, 0, pitched };
        uint32_t maxw = 0;
        for (const TileDesc& t : P.tiles) if (t.w > maxw) maxw = t.w;
        // 16 warps per tile when the call has fewer tiles than SMs (shortest band pipeline), 8 up to a few per SM; beyond
        // that one warp per tile: bands of a tile depend on each other, so extra warps only wait on the band above, and
        // with thousands of tiles the tiles themselves are the parallelism
        uint32_t nw = call_tiles <= 148 ? 16u : (call_tiles <= ctx->root->unr_multi_max_tiles ? 8u : 1u);
        if (pitched) {   // batches: one warp per RGB tile on the row-pitched residual plane; whatever it cannot take goes on below
            LAUNCH(k_dec_unpredict_rgb, ntiles, 32, 0, ua);
            if (all_pitched) nw = 0;
        }
        if (nw == 0) { }
        else if (nw == 16) LAUNCH(k_dec_unpredict_rows<16>, ntiles, 16 * 32, 16 * 2 * 32 * UNR_PITCH, ua);
        else if (nw == 8) LAUNCH(k_dec_unpredict_rows<8>, ntiles, 8 * 32, 8 * 2 * 32 * UNR_PITCH, ua);
        else LAUNCH(k_dec_unpredict_rows<1>, ntiles, 32, 2 * 32 * UNR_PITCH, ua);
        ua.min_w = UNR_MAXW;
        if (maxw > UNR_MAXW) LAUNCH(k_dec_unpredict, ntiles, UNP_THREADS, 0, ua);   // very wide, flat tiles only
        if (any2) LAUNCH(k_dec_grey_raw, ntiles, 256, 0, d_tiles, d_imgs, (const DecTile*)d_dt, din);
    }
    if (any7 && !sel) LAUNCH(k_load7, dim3(296, n), 256, 0, (const ImageDesc*)ctx->imgs.p, (const uint64_t*)ctx->offs.p, din);   // stored images: flat copies
    if (ntiles) LAUNCH(k_dec_copy, ntiles, 256, 0, d_tiles, d_imgs, (const DecTile*)d_dt, din, (uint8_t*)nullptr);
    if (!crops.empty()) {   // one warp per row; enough row blocks that a single large crop fills the machine
        uint32_t maxrows = 0;
        for (const CropDesc& c : crops) if (c.rows > maxrows) maxrows = c.rows;
        const unsigned gx = (maxrows + 7) / 8 < 296 ? (maxrows + 7) / 8 : 296;
        for (size_t c0 = 0; c0 < crops.size(); c0 += 65535) {   // grid y limit
            const unsigned m = (unsigned)(crops.size() - c0 < 65535 ? crops.size() - c0 : 65535);
            LAUNCH(k_crop_rows, dim3(gx, m), 256, 0, (const CropDesc*)ctx->crops.p + c0);
        }
    }
    if (!odescs.empty()) LAUNCH(k_orient, (unsigned)octas, 256, 0, (const OrientDesc*)ctx->orients.p, (uint32_t)odescs.size());
    if (!rdescs.empty()) {   // windows and weights, then the two passes, in Pillow's order for most entries
        const ResizeDesc* d_rd = (const ResizeDesc*)ctx->rdescs.p;
        const uint32_t nr = (uint32_t)rdescs.size();
        bool vfirst = false;   // a chunk with a vertical-first entry gets a vertical launch before the horizontal one too
        for (const ResizeDesc& d : rdescs) vfirst |= d.kx && d.ky && d.h.last;
        LAUNCH(k_resize_coeffs, (unsigned)((rcoef + 255) / 256), 256, 0, d_rd, nr, (uint32_t)rcoef);
        if (vfirst && rv) LAUNCH(k_resize_v, (unsigned)rv, RV_X, 0, d_rd, nr, 1u);
        if (rh) LAUNCH(k_resize_h, (unsigned)rh, RH_X, 0, d_rd, nr);
        if (rv) LAUNCH(k_resize_v, (unsigned)rv, RV_X, 0, d_rd, nr, vfirst ? 2u : 3u);
    }
    for (uint32_t k = 0; k < anstage; k++) {   // augment step k of every entry that has one, before the colour
        uint8_t* const ad = (uint8_t*)ctx->adescs.p;
        if (!apix[k].empty()) LAUNCH(k_aug_pix, (unsigned)apctas[k], AP_THREADS, 0, (const AugPix*)(ad + aat[k].pix), (uint32_t)apix[k].size());
        if (!acol[k].empty()) {
            const ColorDesc* d_cd = (const ColorDesc*)(ad + aat[k].col);
            unsigned long long* d_sum = (unsigned long long*)(ad + adesc_bytes + aat[k].sum);
            if (amctas[k]) LAUNCH(k_color_mean, (unsigned)amctas[k], 256, 0, d_cd, (uint32_t)acol[k].size(), d_sum);
            LAUNCH(k_color, (unsigned)acctas[k], 256, 0, d_cd, (uint32_t)acol[k].size(), (const unsigned long long*)d_sum);
        }
        if (!alut[k].empty()) {
            AugLut* d_al = (AugLut*)(ad + aat[k].lut);
            if (ahctas[k]) {
                LAUNCH(k_aug_hist, (unsigned)ahctas[k], 256, 0, d_al, (uint32_t)alut[k].size());
                LAUNCH(k_aug_lut_build, (unsigned)alut[k].size(), 256, 0, d_al);
            }
            LAUNCH(k_aug_lut, (unsigned)alctas[k], 256, 0, d_al, (uint32_t)alut[k].size());
        }
    }
    if (!cdescs.empty()) {   // the contrast means first, then every coloured entry's chain
        const ColorDesc* d_cd = (const ColorDesc*)ctx->cdescs.p;
        unsigned long long* d_sum = (unsigned long long*)((uint8_t*)ctx->cdescs.p + csum);
        if (mctas) LAUNCH(k_color_mean, (unsigned)mctas, 256, 0, d_cd, (uint32_t)cdescs.size(), d_sum);
        LAUNCH(k_color, (unsigned)cctas, 256, 0, d_cd, (uint32_t)cdescs.size(), (const unsigned long long*)d_sum);
    }
    for (uint32_t k = 0, at = 0; k < nstage; at += (uint32_t)bstage[k].size(), k++)   // after the colour, pass stage by stage
        LAUNCH(k_blur, (unsigned)bctas[k], BL_THREADS, 0, (const BlurPass*)ctx->bdescs.p + at, (uint32_t)bstage[k].size());
    if (!tdescs.empty()) LAUNCH(k_to_tensor, (unsigned)tctas, 256, 0, (const TensorDesc*)ctx->tdescs.p, (uint32_t)tdescs.size(), *fmt);
    // the error flag travels to pinned memory behind the DecImage table
    CK(cudaMemcpyAsync((uint8_t*)ctx->pin_b.p + n * (sizeof(DecImage) + 8), d_err, 4, cudaMemcpyDeviceToHost, ctx->stream));
    return 0;
}

// Entries with equal (file_offsets[i], file_sizes[i]) read one file.  When some file is read by several entries, ord gets
// the entries group by group (ord[p]: the caller's index of position p; groups in the order of their first entry, entries
// in the caller's order), first[p] marks where a group starts, and share[p] says how position p is decoded (Share).
// Otherwise all three stay empty and the call runs in the caller's order, each entry on its own.
static void group_entries(const xpngb_image* imgs, const RegionSel* sel, const uint64_t* file_offsets, const uint64_t* file_sizes,
                          uint32_t n, std::vector<uint32_t>& ord, std::vector<uint8_t>& first, std::vector<Share>& share) {
    std::map<std::pair<uint64_t, uint64_t>, uint32_t> key;
    std::vector<uint32_t> gof(n), start;   // group of each entry; entries per group, then where each group starts
    for (uint32_t i = 0; i < n; i++) {
        const auto it = key.emplace(std::make_pair(file_offsets[i], file_sizes[i]), (uint32_t)start.size());
        if (it.second) start.push_back(0);
        gof[i] = it.first->second;
        start[gof[i]]++;
    }
    if (start.size() == n) return;
    const uint32_t ng = (uint32_t)start.size();
    std::vector<uint32_t> cnt(start);
    for (uint32_t g = 0, at = 0; g < ng; g++) { const uint32_t c = start[g]; start[g] = at; at += c; }
    ord.resize(n); first.assign(n, 0); share.assign(n, Share{ 1, {}, {} });
    std::vector<uint32_t> fill(start);
    for (uint32_t i = 0; i < n; i++) ord[fill[gof[i]]++] = i;
    for (uint32_t g = 0; g < ng; g++) {
        const uint32_t p0 = start[g], i0 = ord[p0];
        first[p0] = 1;
        if (cnt[g] == 1 || imgs[i0].mode == 7) continue;   // stored rectangles are read straight out of the file
        TileSel s = sel[i0].s;
        for (uint32_t p = p0 + 1; p < p0 + cnt[g]; p++) {
            const TileSel& t = sel[ord[p]].s;
            if (t.r0 < s.r0) s.r0 = t.r0; if (t.r1 > s.r1) s.r1 = t.r1;
            if (t.c0 < s.c0) s.c0 = t.c0; if (t.c1 > s.c1) s.c1 = t.c1;
            share[p].n = 0;
        }
        const TileGrid& gr = sel[i0].g;
        share[p0] = Share{ cnt[g], s, xpngb_rect{ gr.x_of(s.c0), gr.y_of(s.r0), gr.x_of(s.c1) + gr.w_of(s.c1) - gr.x_of(s.c0),
                                                  gr.y_of(s.r1) + gr.h_of(s.r1) - gr.y_of(s.r0) } };
    }
}

// The host copies of a call, [a, b) byte ranges each owned by one chunk: sorted by start, neighbouring ranges of one chunk
// become one copy.  So a chunk's copy never spans bytes another chunk copies (its outputs, written back by another lane,
// perhaps later), and a file read by several entries of one chunk crosses PCIe once.  Returns each chunk's copies.
struct Span { uint64_t a, b; uint32_t chunk; };
static std::vector<std::vector<std::pair<uint64_t, uint64_t>>> copy_runs(std::vector<Span>& s, uint32_t nchunks) {
    std::sort(s.begin(), s.end(), [](const Span& x, const Span& y) { return x.a < y.a || (x.a == y.a && x.chunk < y.chunk); });
    std::vector<std::vector<std::pair<uint64_t, uint64_t>>> runs(nchunks);
    for (size_t k = 0; k < s.size(); k++) {
        auto& r = runs[s[k].chunk];
        if (k && s[k - 1].chunk == s[k].chunk && !r.empty()) { if (s[k].b > r.back().second) r.back().second = s[k].b; }
        else r.emplace_back(s[k].a, s[k].b);
    }
    return runs;
}

// xpngb_decode (rects == nullptr), xpngb_decode_region and, with ops, xpngb_decode_oriented; with sizes
// xpngb_decode_resized, with fmt xpngb_decode_tensor, with filters or windows (only with sizes) xpngb_decode_resampled.
// An oriented, resized or tensor call always selects tiles per entry: without rects every entry's rectangle is its whole
// image.  With colors, xpngb_decode_color.
static int decode_call(xpngb_ctx* ctx, xpngb_image* imgs, const xpngb_rect* rects, const int* ops, const xpngb_size* sizes,
                       const int* filters, const xpngb_rect* windows, const xpngb_tensor* fmt, const xpngb_color* colors,
                       const xpngb_blur* blurs, const xpngb_augment* augs, uint32_t n, const void* files,
                       uint64_t files_size, int files_on_device, const uint64_t* file_offsets, const uint64_t* file_sizes, void* pixels,
                       uint64_t pixels_cap, int pixels_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0; ctx->launches = 0; ctx->decoded_tiles = 0; ctx->last_ms = 0.f; ctx->cur = ctx->stream;
    if (!imgs || !files || !file_offsets || !file_sizes || !pixels) FAIL("null argument");
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    for (uint32_t i = 0; i < n; i++) {
        if (file_sizes[i] < 11 || file_sizes[i] > files_size || file_offsets[i] > files_size - file_sizes[i]) FAIL("file %u: bad offset/size", i);
        if (ops && (ops[i] < OP_R90 || ops[i] > OP_TR)) FAIL("entry %u: unknown orientation op %d", i, ops[i]);
        if (sizes && (!sizes[i].w || !sizes[i].h || sizes[i].w > (1u << 24) || sizes[i].h > (1u << 24)))
            FAIL("entry %u: output size %ux%u is not in 1..2^24 on each side", i, sizes[i].w, sizes[i].h);
        if (filters && resize_support((uint32_t)filters[i]) == 0.0)
            FAIL("entry %u: unknown resampling filter %d (LANCZOS 1, BILINEAR 2, BICUBIC 3, BOX 4, HAMMING 5; NEAREST is not one)", i, filters[i]);
        const xpngb_rect* wr = windows ? windows + i : nullptr;
        if (wr && (!wr->w || !wr->h || wr->x >= sizes[i].w || wr->w > sizes[i].w - wr->x || wr->y >= sizes[i].h || wr->h > sizes[i].h - wr->y))
            FAIL("entry %u: window (%llu, %llu) %llux%llu is empty or not inside the %ux%u resized image", i, (unsigned long long)wr->x,
                 (unsigned long long)wr->y, (unsigned long long)wr->w, (unsigned long long)wr->h, sizes[i].w, sizes[i].h);
        if (colors) {
            const xpngb_color& c = colors[i];
            uint32_t seen = 0;
            for (int k = 0; k < 4; k++) seen |= c.order[k] < 4 ? 1u << c.order[k] : 16u;
            if (seen != 15u) FAIL("entry %u: colour order (%u, %u, %u, %u) is not a permutation of 0..3", i, c.order[0], c.order[1],
                                  c.order[2], c.order[3]);
            if (c.on & ~15u) FAIL("entry %u: colour steps 0x%x set a bit above 3", i, c.on);
            if (c.gray > 1) FAIL("entry %u: gray %u is neither 0 nor 1", i, c.gray);
            static const char* const step_name[3] = { "brightness", "contrast", "saturation" };
            for (int k = 0; k < 3; k++)   // Pillow narrows the factor to a float: it must stay finite there too
                if (!(c.factor[k] >= 0.0 && c.factor[k] <= 3.4028234663852886e38))
                    FAIL("entry %u: %s factor %g is negative or not finite", i, step_name[k], c.factor[k]);
            if (!(c.factor[XPNGB_CJ_HUE] >= -0.5 && c.factor[XPNGB_CJ_HUE] <= 0.5))
                FAIL("entry %u: hue factor %g is not in [-0.5, 0.5]", i, c.factor[XPNGB_CJ_HUE]);
        }
        if (blurs) {
            const xpngb_blur& b = blurs[i];
            for (int a = 0; a < 2; a++) {
                if (!(b.radius[a] >= 0.0 && b.radius[a] <= 1.7976931348623157e308))
                    FAIL("entry %u: blur radius %g is negative or not finite", i, b.radius[a]);
                if ((float)b.radius[a] > (float)XPNGB_BLUR_RADIUS_MAX)   // Pillow narrows the radius to a float
                    FAIL("entry %u: blur radius %.9g is above %.0f, where Pillow's uint32 box sums wrap", i, b.radius[a],
                         XPNGB_BLUR_RADIUS_MAX);
            }
            if (b.solarize > 1) FAIL("entry %u: solarize %u is neither 0 nor 1", i, b.solarize);
            if (b.threshold != b.threshold) FAIL("entry %u: solarize threshold is NaN", i);
        }
        if (augs) {
            const xpngb_augment& A = augs[i];
            if (A.nsteps > XPNGB_AUG_STEPS_MAX) FAIL("entry %u: %u augment steps, above %d", i, A.nsteps, XPNGB_AUG_STEPS_MAX);
            for (uint32_t k = 0; k < A.nsteps; k++) {
                const xpngb_aug_step& s = A.step[k];
                if (s.kind > XPNGB_AUG_INVERT) FAIL("entry %u: augment step %u has unknown kind %u", i, k, s.kind);
                if (s.kind == XPNGB_AUG_AFFINE) {
                    if (s.arg != 0 && s.arg != 2 && s.arg != 3)
                        FAIL("entry %u: augment step %u has unknown resample %d (NEAREST 0, BILINEAR 2, BICUBIC 3)", i, k, s.arg);
                    for (int c = 0; c < 6; c++)   // below 2^64 no running sum or product of Pillow's can reach infinity
                        if (!(fabs(s.data[c]) < 18446744073709551616.0))
                            FAIL("entry %u: augment step %u matrix coefficient %g is not finite or not below 2^64", i, k, s.data[c]);
                }
                if (s.kind == XPNGB_AUG_TRANSPOSE && (s.arg < OP_R90 || s.arg > OP_TR))
                    FAIL("entry %u: augment step %u transpose %d is not an op code", i, k, s.arg);
                if (s.kind >= XPNGB_AUG_BRIGHTNESS && s.kind <= XPNGB_AUG_SHARPNESS && !(s.value >= 0.0 && s.value <= 3.4028234663852886e38))
                    FAIL("entry %u: augment step %u factor %g is negative or not finite", i, k, s.value);   // Pillow narrows it to a float
                if (s.kind == XPNGB_AUG_POSTERIZE && (s.arg < 0 || s.arg > 8))
                    FAIL("entry %u: augment step %u posterize bits %d are not in 0..8", i, k, s.arg);
                if (s.kind == XPNGB_AUG_SOLARIZE && s.value != s.value) FAIL("entry %u: augment step %u solarize threshold is NaN", i, k);
            }
        }
    }
    const uint8_t* din = (const uint8_t*)files;
    if (!files_on_device) { ENSURE(files, files_size); din = (const uint8_t*)ctx->files.p; }
    // ---- headers (libxpng.c:969-973)
    std::vector<uint32_t> hdr(2 * n);
    if (!files_on_device) {
        for (uint32_t i = 0; i < n; i++) memcpy(&hdr[2 * i], (const uint8_t*)files + file_offsets[i], 8);
    } else {
        ENSURE(offs, n * 8); ENSURE(hdr, n * 8);
        if (ensure_pin(ctx, ctx->pin_a, n * 8)) return 1;
        memcpy(ctx->pin_a.p, file_offsets, n * 8);
        CK(cudaMemcpyAsync(ctx->offs.p, ctx->pin_a.p, n * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(k_gather_headers, (n + 127) / 128, 128, 0, din, (const uint64_t*)ctx->offs.p, n, (uint32_t*)ctx->hdr.p);
        CK(cudaMemcpyAsync(hdr.data(), ctx->hdr.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    // ---- every entry is checked before anything is decoded
    std::vector<DecImage> DI(n);
    const bool use_sel = rects || ops || sizes || fmt || colors || blurs || augs;
    std::vector<RegionSel> sel(use_sel ? n : 0);
    for (uint32_t i = 0; i < n; i++) {
        if (decode_check(ctx, i, imgs[i], &hdr[2 * i], file_offsets[i], file_sizes[i], rects ? rects + i : nullptr, sizes ? sizes + i : nullptr,
                         windows ? windows + i : nullptr, fmt, pixels_cap, DI[i])) return 1;
        if (colors && colors[i].gray && imgs[i].A && (!fmt || fmt->channels == 0))
            FAIL("entry %u: grayscale of an RGBA entry whose output keeps alpha (torchvision's RandomGrayscale refuses 4 channels)", i);
        if (blurs && blurs[i].solarize && imgs[i].A && (!fmt || fmt->channels == 0))
            FAIL("entry %u: solarize of an RGBA entry whose output keeps alpha (ImageOps.solarize refuses RGBA)", i);
        if (augs && augs[i].nsteps && imgs[i].A && (!fmt || fmt->channels == 0))
            FAIL("entry %u: augment of an RGBA entry whose output keeps alpha (Pillow's ImageOps refuse RGBA)", i);
        if (use_sel) {
            RegionSel& R = sel[i];
            R.rect = rects ? rects[i] : xpngb_rect{ 0, 0, imgs[i].w, imgs[i].h };
            if (sizes) {
                R.crop = R.rect; R.full = sizes[i];
                R.win = windows ? windows[i] : xpngb_rect{ 0, 0, sizes[i].w, sizes[i].h };
                R.filter = filters ? (uint32_t)filters[i] : (uint32_t)RF_BILINEAR;
                const bool rx = R.crop.w != R.full.w, ry = R.crop.h != R.full.h;
                R.rs = rx || ry;
                const uint64_t side_max = resize_side_max(R.filter);
                if ((rx && R.crop.w > side_max) || (ry && R.crop.h > side_max))
                    FAIL("entry %u: a crop side above %llu pixels cannot be resized with filter %u", i, (unsigned long long)side_max, R.filter);
                // the decoded rectangle: the span the window's support reaches on a resampled axis, the window itself on
                // an identity axis (an entry with no resampled axis is a plain crop of the window)
                uint64_t x0 = R.win.x, x1 = R.win.x + R.win.w, y0 = R.win.y, y1 = R.win.y + R.win.h;
                if (rx) resize_span(R.filter, R.crop.w, R.full.w, R.win.x, R.win.x + R.win.w, x0, x1);
                if (ry) resize_span(R.filter, R.crop.h, R.full.h, R.win.y, R.win.y + R.win.h, y0, y1);
                R.rect = xpngb_rect{ R.crop.x + x0, R.crop.y + y0, x1 - x0, y1 - y0 };
            }
            region_select(imgs[i].w, imgs[i].h, R.rect, R.g, R.s, R.cover);
            const uint64_t ow = sizes ? R.win.w : R.rect.w, oh = sizes ? R.win.h : R.rect.h;
            for (uint32_t k = 0; augs && k < augs[i].nsteps; k++) {
                const xpngb_aug_step& s = augs[i].step[k];
                if (s.kind == XPNGB_AUG_TRANSPOSE && (s.arg == OP_R90 || s.arg == OP_R270) && ow != oh)
                    FAIL("entry %u: augment step %u turns a %llux%llu output a quarter (Image.rotate does that for squares only)", i, k,
                         (unsigned long long)ow, (unsigned long long)oh);
            }
        }
    }
    uint8_t* dpx = (uint8_t*)pixels;
    if (!pixels_on_device) { ENSURE(pixels, pixels_cap); dpx = (uint8_t*)ctx->pixels.p; }
    // ---- entries that read the same file decode it once; the chunks then see them group by group, position p being
    // the caller's entry at(p)
    std::vector<uint32_t> ord;
    std::vector<uint8_t> first;
    std::vector<Share> share;
    if (use_sel) group_entries(imgs, sel.data(), file_offsets, file_sizes, n, ord, first, share);
    auto at = [&](uint32_t p) { return ord.empty() ? p : ord[p]; };
    auto permuted = [&](auto* a, auto& v) -> decltype(a) {   // a in position order (a itself when nothing is reordered)
        if (!a || ord.empty()) return a;
        v.reserve(n);
        for (uint32_t p = 0; p < n; p++) v.push_back(a[ord[p]]);
        return v.data();
    };
    std::vector<xpngb_image> o_imgs; std::vector<DecImage> o_DI; std::vector<RegionSel> o_sel; std::vector<int> o_ops;
    std::vector<xpngb_color> o_colors; std::vector<xpngb_blur> o_blurs; std::vector<xpngb_augment> o_augs;
    const xpngb_image* p_imgs = permuted((const xpngb_image*)imgs, o_imgs);
    const DecImage* p_DI = permuted((const DecImage*)DI.data(), o_DI);
    const RegionSel* p_sel = use_sel ? permuted((const RegionSel*)sel.data(), o_sel) : nullptr;
    const int* p_ops = permuted(ops, o_ops);
    const xpngb_color* p_colors = permuted(colors, o_colors);
    const xpngb_blur* p_blurs = permuted(blurs, o_blurs);
    const xpngb_augment* p_augs = permuted(augs, o_augs);
    // chunks are cut by the pixels each position decodes: the whole image, the cover of its rectangle (stored: the
    // rectangle), or for a shared window its cover at the group's first position and nothing at the others
    std::vector<xpngb_image> dims(n);
    uint64_t tiles_est = 0; bool l2 = false;
    for (uint32_t p = 0; p < n; p++) {
        const uint32_t i = at(p), mode = imgs[i].mode;
        const bool sh = !share.empty() && share[p].n != 1;
        const xpngb_rect none{};
        const xpngb_rect* wh = !use_sel ? nullptr : mode == 7 ? &sel[i].rect : !sh ? &sel[i].cover : share[p].n ? &share[p].cover : &none;
        const TileSel& s = sh ? share[p].s : use_sel ? sel[i].s : TileSel{};
        dims[p].w = wh ? wh->w : imgs[i].w; dims[p].h = wh ? wh->h : imgs[i].h;
        if ((mode == 1 || mode == 2) && !(sh && !share[p].n))
            tiles_est += use_sel ? (s.r1 - s.r0 + 1) * (s.c1 - s.c0 + 1) : (imgs[i].w * imgs[i].h + TILE_AREA - 1) / TILE_AREA;
        l2 |= mode == 2;
    }
    auto out_bytes = [&](uint32_t i) {
        return entry_out_bytes(imgs[i], rects ? rects + i : nullptr, sizes ? sizes + i : nullptr, windows ? windows + i : nullptr, fmt);
    };
    // level 2: above ~600 tiles the pair family wins, with the 16-symbol value streams warp-per-block while they all fit
    // (s16_lat_max_tiles); level 1: the warp-per-block family up to ~1300 tiles (measured at 125 / 250 / 500 frames, profiles/)
    const bool lat = l2 ? 17 * tiles_est <= (uint64_t)ctx->lat_max_blocks * 5 / 6 : 9 * tiles_est <= ctx->lat_max_blocks;
    const std::vector<uint32_t> cuts = cut_chunks(ctx, dims.data(), n, first.empty() ? nullptr : first.data());
    const uint32_t nchunks = (uint32_t)cuts.size() - 1;
    std::vector<Span> fspan, ospan;
    for (uint32_t ci = 0; ci < nchunks; ci++)
        for (uint32_t p = cuts[ci]; p < cuts[ci + 1]; p++) {
            const uint32_t i = at(p);
            if (!files_on_device) fspan.push_back(Span{ file_offsets[i], file_offsets[i] + file_sizes[i], ci });
            if (!pixels_on_device) ospan.push_back(Span{ imgs[i].offset, imgs[i].offset + out_bytes(i), ci });
        }
    const auto uploads = copy_runs(fspan, nchunks), downloads = copy_runs(ospan, nchunks);
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    int rc = 0;
    std::vector<xpngb_ctx*> used(nchunks, nullptr);
    std::vector<uint32_t> cn(nchunks, 0);
    auto chunk_done = [&](uint32_t ci) -> int {   // wait for chunk ci, read its error flag
        xpngb_ctx* lane = used[ci];
        CK(cudaStreamSynchronize(lane->stream));
        int herr = 0; memcpy(&herr, (uint8_t*)lane->pin_b.p + cn[ci] * (sizeof(DecImage) + 8), 4);
        if (herr) FAIL("corrupt .xpng data (decoder error %d)", herr);
        return 0;
    };
    uint32_t done = 0;
    for (uint32_t ci = 0; ci < nchunks && !rc; ci++) {
        const uint32_t li = ci % ctx->pipe_lanes;
        while (!rc && ci >= ctx->pipe_lanes && done <= ci - ctx->pipe_lanes) rc = chunk_done(done++);
        if (rc) break;
        xpngb_ctx* lane = lane_get(ctx, li);
        if (!lane) { snprintf(ctx->err, sizeof ctx->err, "cannot create pipeline lane %u", li); rc = 1; break; }
        used[ci] = lane; cn[ci] = cuts[ci + 1] - cuts[ci];
        const uint32_t i0 = cuts[ci], m = cn[ci];
        if (lane != ctx && cudaStreamWaitEvent(lane->stream, ctx->ev0, 0) != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "cudaStreamWaitEvent failed"); rc = 1; break; }
        for (const auto& r : uploads[ci])
            if (cudaMemcpyAsync((uint8_t*)ctx->files.p + r.first, (const uint8_t*)files + r.first, r.second - r.first, cudaMemcpyHostToDevice,
                                lane->stream) != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "host to device copy failed"); rc = 1; break; }
        if (rc) break;
        rc = decode_issue(lane, lat, p_imgs + i0, p_DI + i0, p_sel ? p_sel + i0 : nullptr, share.empty() ? nullptr : share.data() + i0,
                          p_ops ? p_ops + i0 : nullptr, fmt, p_colors ? p_colors + i0 : nullptr, p_blurs ? p_blurs + i0 : nullptr,
                          p_augs ? p_augs + i0 : nullptr, m, din, dpx, (uint32_t)(tiles_est > 0xFFFFFFFFull ? 0xFFFFFFFFu : tiles_est));
        for (size_t k = 0; !rc && k < downloads[ci].size(); k++) {
            const auto& r = downloads[ci][k];
            if (cudaMemcpyAsync((uint8_t*)pixels + r.first, dpx + r.first, r.second - r.first, cudaMemcpyDeviceToHost, lane->stream) != cudaSuccess) {
                snprintf(ctx->err, sizeof ctx->err, "device to host copy failed"); rc = 1;
            }
        }
    }
    // every issued chunk is waited for, also after an error (the caller's buffers must be quiet when we return)
    for (; done < nchunks; done++) {
        if (!used[done]) continue;
        if (rc) cudaStreamSynchronize(used[done]->stream);
        else rc = chunk_done(done);
    }
    for (uint32_t li = 1; li <= ctx->lanes.size(); li++) {
        xpngb_ctx* lane = ctx->lanes[li - 1];
        cudaEventRecord(lane->ev_done, lane->stream);
        cudaStreamWaitEvent(ctx->stream, lane->ev_done, 0);
    }
    cudaEventRecord(ctx->ev1, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    if (rc) return 1;
    CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
    tl_dump(ctx, "dec");
    return 0;
}

extern "C" int xpngb_decode(xpngb_ctx* ctx, xpngb_image* imgs, uint32_t n, const void* files, uint64_t files_size, int files_on_device,
                            const uint64_t* file_offsets, const uint64_t* file_sizes, void* pixels, uint64_t pixels_cap,
                            int pixels_on_device) {
    return decode_call(ctx, imgs, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes, pixels, pixels_cap,
                       pixels_on_device);
}

extern "C" int xpngb_decode_region(xpngb_ctx* ctx, xpngb_image* imgs, const xpngb_rect* rects, uint32_t n, const void* files,
                                   uint64_t files_size, int files_on_device, const uint64_t* file_offsets, const uint64_t* file_sizes,
                                   void* pixels, uint64_t pixels_cap, int pixels_on_device) {
    if (!ctx) return 1;
    if (!rects) { ctx->err[0] = 0; FAIL("null argument"); }
    return decode_call(ctx, imgs, rects, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes, pixels, pixels_cap,
                       pixels_on_device);
}

extern "C" int xpngb_decode_oriented(xpngb_ctx* ctx, const int* ops, xpngb_image* imgs, const xpngb_rect* rects, uint32_t n,
                                     const void* files, uint64_t files_size, int files_on_device, const uint64_t* file_offsets,
                                     const uint64_t* file_sizes, void* pixels, uint64_t pixels_cap, int pixels_on_device) {
    if (!ctx) return 1;
    if (!ops) { ctx->err[0] = 0; FAIL("null argument"); }
    return decode_call(ctx, imgs, rects, ops, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes, pixels, pixels_cap,
                       pixels_on_device);
}

extern "C" int xpngb_decode_resized(xpngb_ctx* ctx, const int* ops, xpngb_image* imgs, const xpngb_rect* rects, const xpngb_size* sizes,
                                    uint32_t n, const void* files, uint64_t files_size, int files_on_device, const uint64_t* file_offsets,
                                    const uint64_t* file_sizes, void* pixels, uint64_t pixels_cap, int pixels_on_device) {
    if (!ctx) return 1;
    if (!sizes) { ctx->err[0] = 0; FAIL("null argument"); }
    return decode_call(ctx, imgs, rects, ops, sizes, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes, pixels, pixels_cap,
                       pixels_on_device);
}

// The format of a tensor decode, checked before anything else.  A float dtype normalises every channel it may write: the
// first 3, or all 4 when alpha is kept (a batch may hold RGBA files).
static int tensor_check(xpngb_ctx* ctx, const xpngb_tensor* f) {
    if (!f) FAIL("null argument (fmt)");
    if (f->dtype > XPNGB_DT_BF16) FAIL("tensor format: unknown dtype %u", f->dtype);
    if (f->layout > XPNGB_HWC) FAIL("tensor format: unknown layout %u", f->layout);
    if (f->scale > XPNGB_SCALE_MUL) FAIL("tensor format: unknown scale %u", f->scale);
    if (f->channels != 0 && f->channels != 3) FAIL("tensor format: channels %u is neither 0 (as stored) nor 3 (RGB)", f->channels);
    if (f->dtype != XPNGB_DT_U8)
        for (uint32_t c = 0; c < (f->channels == 3 ? 3u : 4u); c++) {
            if (!isfinite(f->mean[c])) FAIL("tensor format: mean[%u] is not finite", c);
            if (!isfinite(f->std[c]) || f->std[c] == 0.f) FAIL("tensor format: std[%u] is zero or not finite", c);
        }
    return 0;
}

extern "C" int xpngb_decode_tensor(xpngb_ctx* ctx, const xpngb_tensor* fmt, const int* ops, xpngb_image* imgs, const xpngb_rect* rects,
                                   const xpngb_size* sizes, uint32_t n, const void* files, uint64_t files_size, int files_on_device,
                                   const uint64_t* file_offsets, const uint64_t* file_sizes, void* out, uint64_t out_cap, int out_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0;
    if (tensor_check(ctx, fmt)) return 1;
    return decode_call(ctx, imgs, rects, ops, sizes, nullptr, nullptr, fmt, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes, out, out_cap,
                       out_on_device);
}

extern "C" int xpngb_decode_resampled(xpngb_ctx* ctx, const xpngb_tensor* fmt, const int* filters, const int* ops, xpngb_image* imgs,
                                      const xpngb_rect* rects, const xpngb_size* sizes, const xpngb_rect* windows, uint32_t n,
                                      const void* files, uint64_t files_size, int files_on_device, const uint64_t* file_offsets,
                                      const uint64_t* file_sizes, void* out, uint64_t out_cap, int out_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0;
    if (!sizes) FAIL("null argument (sizes)");
    if (fmt && tensor_check(ctx, fmt)) return 1;
    return decode_call(ctx, imgs, rects, ops, sizes, filters, windows, fmt, nullptr, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets, file_sizes,
                       out, out_cap, out_on_device);
}

extern "C" int xpngb_decode_color(xpngb_ctx* ctx, const xpngb_tensor* fmt, const int* filters, const int* ops, xpngb_image* imgs,
                                  const xpngb_rect* rects, const xpngb_size* sizes, const xpngb_rect* windows, const xpngb_color* colors,
                                  uint32_t n, const void* files, uint64_t files_size, int files_on_device, const uint64_t* file_offsets,
                                  const uint64_t* file_sizes, void* out, uint64_t out_cap, int out_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0;
    if (!sizes && (filters || windows)) FAIL("null argument (sizes): filters and windows need sizes");
    if (fmt && tensor_check(ctx, fmt)) return 1;
    return decode_call(ctx, imgs, rects, ops, sizes, filters, windows, fmt, colors, nullptr, nullptr, n, files, files_size, files_on_device, file_offsets,
                       file_sizes, out, out_cap, out_on_device);
}

extern "C" int xpngb_decode_blur(xpngb_ctx* ctx, const xpngb_tensor* fmt, const int* filters, const int* ops, xpngb_image* imgs,
                                 const xpngb_rect* rects, const xpngb_size* sizes, const xpngb_rect* windows, const xpngb_color* colors,
                                 const xpngb_blur* blurs, uint32_t n, const void* files, uint64_t files_size, int files_on_device,
                                 const uint64_t* file_offsets, const uint64_t* file_sizes, void* out, uint64_t out_cap, int out_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0;
    if (!sizes && (filters || windows)) FAIL("null argument (sizes): filters and windows need sizes");
    if (fmt && tensor_check(ctx, fmt)) return 1;
    return decode_call(ctx, imgs, rects, ops, sizes, filters, windows, fmt, colors, blurs, nullptr, n, files, files_size, files_on_device,
                       file_offsets, file_sizes, out, out_cap, out_on_device);
}

extern "C" int xpngb_decode_augment(xpngb_ctx* ctx, const xpngb_tensor* fmt, const int* filters, const int* ops, xpngb_image* imgs,
                                    const xpngb_rect* rects, const xpngb_size* sizes, const xpngb_rect* windows, const xpngb_color* colors,
                                    const xpngb_blur* blurs, const xpngb_augment* augs, uint32_t n, const void* files, uint64_t files_size,
                                    int files_on_device, const uint64_t* file_offsets, const uint64_t* file_sizes, void* out, uint64_t out_cap,
                                    int out_on_device) {
    if (!ctx) return 1;
    ctx->err[0] = 0;
    if (!sizes && (filters || windows)) FAIL("null argument (sizes): filters and windows need sizes");
    if (fmt && tensor_check(ctx, fmt)) return 1;
    return decode_call(ctx, imgs, rects, ops, sizes, filters, windows, fmt, colors, blurs, augs, n, files, files_size, files_on_device,
                       file_offsets, file_sizes, out, out_cap, out_on_device);
}

extern "C" int xpngb_blur_box(double radius, int32_t* ri, uint32_t* ww, uint32_t* fw) {
    if (!(radius >= 0.0 && radius <= 1.7976931348623157e308) || (float)radius > (float)XPNGB_BLUR_RADIUS_MAX) return 1;
    const BlurBox b = blur_box((float)radius);
    *ri = b.ri; *ww = b.ww; *fw = b.fw;
    return 0;
}

extern "C" uint32_t xpngb_resize_ksize(int filter, uint32_t in, uint32_t out) {
    return in && out ? resize_ksize((uint32_t)filter, in, out) : 0;
}

// The tables k_resize_coeffs computes for output coordinates first .. first + count - 1 of one axis, copied back:
// (xmin, n) pairs and count rows of ksize weights, zero past each window.
extern "C" int xpngb_resize_coeffs(xpngb_ctx* ctx, int filter, uint32_t in, uint32_t out, uint32_t first, uint32_t count,
                                   int32_t* xmin_n, int32_t* k) {
    if (!ctx) return 1;
    ctx->err[0] = 0; ctx->launches = 0; ctx->cur = ctx->stream;
    if (!xmin_n || !k) FAIL("null argument");
    if (resize_support((uint32_t)filter) == 0.0) FAIL("unknown resampling filter %d", filter);
    if (!in || !out || in > (1u << 24) || out > (1u << 24) || in == out) FAIL("in %u, out %u: not a resampled axis", in, out);
    if (!count || first >= out || count > out - first) FAIL("coordinates %u + %u are not inside 0..%u", first, count, out);
    CK(cudaSetDevice(ctx->device));
    ResizeDesc d{};
    d.in_w = in; d.full_w = out; d.out_w = count; d.wx = first; d.filter = (uint32_t)filter;
    d.kx = resize_ksize((uint32_t)filter, in, out);
    const uint64_t tab = resize_table_bytes(count, d.kx);
    ENSURE(rtab, tab); ENSURE(rdescs, sizeof(ResizeDesc));
    d.coef = (uint64_t)ctx->rtab.p;
    CK(cudaMemsetAsync(ctx->rtab.p, 0, tab, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rdescs.p, &d, sizeof d, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_resize_coeffs, (count + 255) / 256, 256, 0, (const ResizeDesc*)ctx->rdescs.p, 1u, count);
    CK(cudaMemcpyAsync(xmin_n, ctx->rtab.p, (uint64_t)count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(k, (uint8_t*)ctx->rtab.p + (uint64_t)count * 8, (uint64_t)count * d.kx * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// YCoCg-R side component
// ------------------------------------------------------------------------------------------------
extern "C" int xpngb_ycocg_forward(xpngb_ctx* ctx, const uint8_t* rgb, int16_t* ycc, uint64_t n) {
    if (!ctx || !rgb || !ycc) return 1;
    CK(cudaSetDevice(ctx->device));
    ENSURE(m2a, 3 * n); ENSURE(m2b, 6 * n);
    CK(cudaMemcpyAsync(ctx->m2a.p, rgb, 3 * n, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_ycocg_fwd, 1184, 256, 0, (const uint8_t*)ctx->m2a.p, (int16_t*)ctx->m2b.p, n);
    CK(cudaMemcpyAsync(ycc, ctx->m2b.p, 6 * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int xpngb_ycocg_inverse(xpngb_ctx* ctx, const int16_t* ycc, uint8_t* rgb, uint64_t n) {
    if (!ctx || !rgb || !ycc) return 1;
    CK(cudaSetDevice(ctx->device));
    ENSURE(m2a, 3 * n); ENSURE(m2b, 6 * n);
    CK(cudaMemcpyAsync(ctx->m2b.p, ycc, 6 * n, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_ycocg_inv, 1184, 256, 0, (const int16_t*)ctx->m2b.p, (uint8_t*)ctx->m2a.p, n);
    CK(cudaMemcpyAsync(rgb, ctx->m2a.p, 3 * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
