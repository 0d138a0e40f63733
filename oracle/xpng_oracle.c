/*
 * xpng_oracle.c — CPU restatement of the xPNG encode/decode hot path (see xpng_oracle.h).
 *
 * TEST INFRASTRUCTURE ONLY: this is the parity checker, never the product path.
 * Written from the format description (SURVEY.md App. A/B) and the behaviour of the reference;
 * citations "ref:" name file:line of /root/reference that each routine restates.
 * Single-threaded, in-memory, little-endian hosts only (like the reference).
 */
#include "xpng_oracle.h"
#include <stdlib.h>
#include <string.h>

#define TILE_AREA (444u * 444u) /* ref: libxpng.c:49 */
#define RANS_L (1ull << 31)     /* ref: libxpng.c:153 */

/* ------------------------------------------------------------------ scalar helpers (App. B) */

static inline uint32_t bitlen(uint32_t v) { return v ? 32u - (uint32_t)__builtin_clz(v) : 0u; } /* ref :19 */
static inline uint32_t zz8(int v) { int s = (int8_t)v; return (uint32_t)((s << 1) ^ (s >> 31)); } /* ref :20 */
static inline int unzz(uint32_t u) { return (int)(u >> 1) ^ -(int)(u & 1); }                   /* ref :21 */
static inline int pred_avg2(int L, int U) { return (L + U + 1) >> 1; }                          /* ref :27 */
static inline int pred_grad3(int L, int U, int UL) { return (3 * L + 3 * U - 2 * UL + 2) >> 2; } /* ref :29 */

static inline uint32_t ld32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline void st32(uint8_t *p, uint32_t v) { memcpy(p, &v, 4); }
static inline uint64_t ld64(const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); return v; }
static inline void st64(uint8_t *p, uint64_t v) { memcpy(p, &v, 8); }

/* ------------------------------------------------------------------ decision log (xo_trace) */

static __thread xo_decision_t *tr_buf;
static __thread uint64_t tr_cap, tr_len;
static __thread uint32_t tr_tile, tr_stream;

void xo_trace(xo_decision_t *buf, uint64_t cap) { tr_buf = buf; tr_cap = buf ? cap : 0; tr_len = 0; tr_tile = tr_stream = 0; }
uint64_t xo_trace_len(void) { return tr_len; }

/* Records past the capacity are counted, not stored, so a caller can retry with a larger buffer. */
static void tr_put(uint32_t kind, uint32_t outcome, uint64_t v0, uint64_t v1, uint64_t v2, uint64_t v3) {
    if (!tr_buf) return;
    if (tr_len < tr_cap) tr_buf[tr_len] = (xo_decision_t){ kind, tr_tile, tr_stream, outcome, { v0, v1, v2, v3 } };
    tr_len++;
}

/* MSB-first bit writer over little-endian 32-bit words (ref: libxpng.c:8-11, :14-17). */
typedef struct { uint64_t acc; uint32_t n; uint8_t *out; } bitw_t;
static inline void bw_put(bitw_t *b, uint32_t c, uint32_t v) {
    b->acc = (b->acc << c) | v; b->n += c;
    if (b->n >= 32) { b->n -= 32; st32(b->out, (uint32_t)(b->acc >> b->n)); b->out += 4; }
}
static inline void bw_end(bitw_t *b) {
    if (b->n > 0) { st32(b->out, (uint32_t)(b->acc << (32 - b->n))); b->out += 4; b->n = 0; }
}

/* MSB-first bit reader; reads past `end` return zero bits (ref: libxpng.c:9, :12, :15-16). */
typedef struct { const uint8_t *base, *end; uint64_t pos; } bitr_t;
static inline uint32_t br_get(bitr_t *b, uint32_t c) {
    uint32_t v = 0;
    while (c) {
        uint64_t w = b->pos >> 5; uint32_t off = (uint32_t)(b->pos & 31), take = 32 - off;
        if (take > c) take = c;
        const uint8_t *p = b->base + 4 * w;
        uint32_t word = (p + 4 <= b->end) ? ld32(p) : 0;
        uint32_t bits = (word >> (32 - off - take)) & (take == 32 ? 0xFFFFFFFFu : ((1u << take) - 1));
        v = (take == 32) ? bits : ((v << take) | bits);
        b->pos += take; c -= take;
    }
    return v;
}

/* ------------------------------------------------------------------ tiling (App. A.2) */

/* ref: libxpng.c:57-66 — sizes along one axis: [first, second, base, base, ...] */
static uint64_t axis_split(uint64_t extent, uint64_t base, uint64_t *first, uint64_t *second) {
    uint64_t n = extent / base, rem = extent % base;
    *first = base + rem; *second = base;
    if (rem > base / 2) { n++; *second = (base + rem) / 2; *first = *second + ((base + rem) & 1); }
    return n;
}

uint64_t xo_tile_grid(uint64_t W, uint64_t H, int pxsz, xo_tile_t *tiles, uint64_t cap) {
    uint64_t nw = 1, nh = 1, w0 = W, w1 = W, wb = W, h0 = H, h1 = H, hb = H;
    (void)pxsz;
    if (W * H > TILE_AREA) { /* ref :57 (s <= TILE*PXSZ  <=>  W*H <= TILE) */
        if (W < 444) { wb = W; hb = TILE_AREA / W; }
        else if (H < 444) { hb = H; wb = TILE_AREA / H; }
        else wb = hb = 444;
        nw = axis_split(W, wb, &w0, &w1);
        nh = axis_split(H, hb, &h0, &h1);
    }
    uint64_t k = 0, y = 0;
    for (uint64_t i = 0; i < nh; i++) {
        uint64_t th = i == 0 ? h0 : (i == 1 ? h1 : hb), x = 0;
        for (uint64_t j = 0; j < nw; j++) {
            uint64_t tw = j == 0 ? w0 : (j == 1 ? w1 : wb);
            if (tiles && k < cap) tiles[k] = (xo_tile_t){ x, y, tw, th };
            k++; x += tw;
        }
        y += th;
    }
    return k;
}

/* ------------------------------------------------------------------ alpha normalisation */

/* ref: libxpng.c:688-721 */
int xo_normalize(const uint8_t *in, uint64_t w, uint64_t h, int A, uint8_t *out, uint64_t *s_out) {
    uint64_t npx = w * h;
    if (!A) { memcpy(out, in, npx * 3); *s_out = npx * 3; return 0; }
    int translucent = 0, dirty = 0;
    for (uint64_t i = 0; i < npx; i++) {
        uint32_t px = ld32(in + 4 * i), a = px >> 24;
        if (a == 0 && px != 0) { dirty = 1; break; }
        if (a != 255) translucent = 1;
    }
    if (dirty) { /* zero the colour of fully transparent pixels, keep alpha */
        for (uint64_t i = 0; i < npx; i++) {
            uint32_t px = ld32(in + 4 * i);
            st32(out + 4 * i, (px >> 24) ? px : 0);
        }
        *s_out = npx * 4; return 1;
    }
    if (translucent) { memcpy(out, in, npx * 4); *s_out = npx * 4; return 1; }
    for (uint64_t i = 0; i < npx; i++) memcpy(out + 3 * i, in + 4 * i, 3); /* opaque: strip alpha */
    *s_out = npx * 3; return 0;
}

/* ------------------------------------------------------------------ predictor selection */

/* ref: libxpng.c:92-140 */
unsigned xo_select_predictor(const uint8_t *t, uint64_t w, uint64_t h, uint64_t bpr, int pxsz) {
    if (w < 4 || h < 4) return 0;
    uint32_t cost[4] = { 0, 0, 0, 0 };
    for (uint64_t j = 0; j < h / 4; j++) {
        for (uint64_t i = 0; i < w / 4; i++) {
            const uint8_t *p = t + (3 + 4 * j) * bpr + (3 + 4 * i) * (uint64_t)pxsz;
            if (pxsz == 4 && p[3] == 0) continue;
            int a[3], g[3];
            for (int c = 0; c < 3; c++) {
                int L = p[c - pxsz], U = p[c - (int64_t)bpr], UL = p[c - (int64_t)bpr - pxsz];
                a[c] = p[c] - pred_avg2(L, U);
                g[c] = p[c] - pred_grad3(L, U, UL);
            }
            cost[0] += bitlen(zz8(a[0]) | zz8(a[1]) | zz8(a[2]));
            cost[1] += bitlen(zz8(a[0] - a[1]) | zz8(a[1]) | zz8(a[2] - a[1]));
            cost[2] += bitlen(zz8(g[0]) | zz8(g[1]) | zz8(g[2]));
            cost[3] += bitlen(zz8(g[0] - g[1]) | zz8(g[1]) | zz8(g[2] - g[1]));
        }
    }
    unsigned m = 0;
    for (unsigned k = 1; k < 4; k++) if (cost[k] < cost[m]) m = k;
    tr_put(XO_D_PRED, m, cost[0], cost[1], cost[2], cost[3]);
    return (unsigned)(pxsz & 4) | m;
}

/* ------------------------------------------------------------------ frequency model + rANS */

typedef struct { uint64_t rcp; uint32_t freq, bias, cmpl, shift; } encsym_t; /* ref :155-158 */

/* ref: libxpng.c:166-182 and :316-329 — scale the cumulative counts to 2^pb, then the "steal"
 * fix-up so that every used symbol keeps a non-zero width.  cum has N+1 entries. */
static void normalise_freqs(uint32_t *F, uint32_t *cum, unsigned N, uint64_t total, int pb) {
    cum[0] = 0;
    for (unsigned i = 0; i < N; i++) cum[i + 1] = cum[i] + F[i];
    for (unsigned i = 1; i <= N; i++) cum[i] = (uint32_t)(((uint64_t)cum[i] << pb) / total);
    for (unsigned i = 0; i < N; i++) {
        if (F[i] && cum[i + 1] == cum[i]) {
            uint32_t best = ~0u; unsigned donor = 0;
            for (unsigned j = 0; j < N; j++) {
                uint32_t wdt = cum[j + 1] - cum[j];
                if (wdt > 1 && wdt < best) { best = wdt; donor = j; }
            }
            if (tr_buf) { /* how many symbols share the smallest width, and the last of them */
                uint32_t ties = 0, last = 0;
                for (unsigned j = 0; j < N; j++) if (cum[j + 1] - cum[j] == best) { ties++; last = j; }
                tr_put(XO_D_STEAL, donor, i, best, ties, last);
            }
            if (donor < i) for (unsigned j = donor + 1; j <= i; j++) cum[j]--;
            else           for (unsigned j = i + 1; j <= donor; j++) cum[j]++;
        }
    }
    for (unsigned i = 0; i < N; i++) F[i] = cum[i + 1] - cum[i];
}

/* ref: libxpng.c:184-213 and :331-360 (ryg-rans Rans64EncSymbolInit) */
static void build_encsyms(encsym_t *e, const uint32_t *F, const uint32_t *cum, unsigned N, int pb) {
    for (unsigned i = 0; i < N; i++) {
        e[i].freq = F[i]; e[i].cmpl = (1u << pb) - F[i];
        if (F[i] < 2) { e[i].rcp = ~0ull; e[i].shift = 0; e[i].bias = cum[i] + (1u << pb) - 1; }
        else {
            uint32_t sh = 0; while (F[i] > (1u << sh)) sh++;
            /* ceil(2^(sh+63) / freq) */
            unsigned __int128 num = ((unsigned __int128)1 << (sh + 63)) + (F[i] - 1);
            e[i].rcp = (uint64_t)(num / F[i]); e[i].shift = sh - 1; e[i].bias = cum[i];
        }
    }
}

static inline uint64_t rans_put(uint64_t x, const encsym_t *s) { /* ref :375-376 */
    uint64_t q = (uint64_t)(((unsigned __int128)x * s->rcp) >> 64);
    return x + s->bias + (q >> s->shift) * s->cmpl;
}
static inline uint64_t rans_limit(const encsym_t *s, int pb) { /* ref :370 */
    return ((RANS_L >> pb) << 32) * s->freq;
}

/* ref: libxpng.c:396-414 — frequency table as a bit stream; sparse form: 0 | 1+F. */
static void put_freq_table(bitw_t *b, const uint32_t *F, unsigned N, int pb, int sparse, int v1) {
    (void)v1;
    for (unsigned i = 0; i < N; i++) {
        if (!sparse) bw_put(b, (uint32_t)pb, F[i]);
        else if (F[i]) bw_put(b, (uint32_t)pb + 1, F[i] + (1u << pb));
        else bw_put(b, 1, 0);
    }
}

/* ref: libxpng.c:307-427 */
uint64_t xo_block_v2_encode(uint32_t *F, unsigned nsym, const uint8_t *in, uint64_t n,
                            uint8_t *out, int pb) {
    if (n == 0) { st32(out, 4); return 4; }
    int top = (int)nsym; while (F[--top] == 0) {}
    unsigned N = (unsigned)top + 1, used = 0; uint32_t nbit = bitlen((uint32_t)top);
    for (unsigned i = 0; i < N; i++) used += F[i] != 0;
    if (used == 1) { st32(out, 8u | (1u << 24)); st32(out + 4, (uint32_t)n | ((uint32_t)in[0] << 24)); return 8; }

    uint32_t cum[257]; encsym_t e[256];
    normalise_freqs(F, cum, N, n, pb);
    build_encsyms(e, F, cum, N, pb);

    uint8_t *wp = out + 12; uint64_t x0 = RANS_L, x1 = RANS_L, i = 0;
    for (; i + 1 < n; i += 2) { /* forward, two interleaved states (ref :362-380) */
        const encsym_t *s0 = e + in[i], *s1 = e + in[i + 1];
        if (x0 >= rans_limit(s0, pb)) { st32(wp, (uint32_t)x0); wp += 4; x0 >>= 32; }
        if (x1 >= rans_limit(s1, pb)) { st32(wp, (uint32_t)x1); wp += 4; x1 >>= 32; }
        x0 = rans_put(x0, s0); x1 = rans_put(x1, s1);
    }
    if (n & 1) { /* ref :382-392 */
        const encsym_t *s0 = e + in[i];
        if (x0 >= rans_limit(s0, pb)) { st32(wp, (uint32_t)x0); wp += 4; x0 >>= 32; }
        x0 = rans_put(x0, s0);
    }
    st64(wp, x0); st64(wp + 8, x1); wp += 16; /* ref :394 */

    int sparse = (N + used * (unsigned)pb) < N * (unsigned)pb; /* ref :396-397 */
    tr_put(XO_D_V2_TABLE, (uint32_t)sparse, N + used * (unsigned)pb, N * (unsigned)pb, used, N);
    st32(out + 4, (uint32_t)n | ((N - 2) << 24));
    st32(out + 8, (uint32_t)((wp - (out + 8)) / 4) | ((uint32_t)pb << 24)); /* ref :400 */
    bitw_t b = { 0, 0, wp };
    put_freq_table(&b, F, N, pb, sparse, 0); bw_end(&b);
    uint64_t csz = (uint64_t)(b.out - out);
    st32(out, (uint32_t)csz | ((uint32_t)(3 + sparse) << 24));

    uint64_t rawbits = (uint64_t)nbit * n, rawsz = 8 + (rawbits / 32) * 4 + (rawbits % 32 ? 4 : 0);
    tr_put(XO_D_V2_BLOCK, csz < rawsz, csz, rawsz, n, N);
    if (csz >= rawsz) { /* ref :417-424: plain nbit-wide symbols */
        out[7] = (uint8_t)nbit;
        bitw_t r = { 0, 0, out + 8 };
        for (uint64_t k = 0; k < n; k++) bw_put(&r, nbit, in[k]);
        bw_end(&r);
        csz = (uint64_t)(r.out - out);
        st32(out, (uint32_t)csz | (2u << 24));
    }
    return csz;
}

/* Read a frequency table written by put_freq_table (ref :280-281, :453-462). */
static void get_freq_table(bitr_t *b, uint32_t *F, unsigned N, int pb, int sparse) {
    for (unsigned i = 0; i < N; i++) {
        if (!sparse) F[i] = br_get(b, (uint32_t)pb);
        else F[i] = br_get(b, 1) ? br_get(b, (uint32_t)pb) : 0;
    }
}

static void build_slot_table(uint8_t *slot2sym, uint32_t *cum, const uint32_t *F, unsigned N, int pb) {
    cum[0] = 0;
    for (unsigned i = 0; i < N; i++) cum[i + 1] = cum[i] + F[i];
    for (unsigned i = 0; i < N; i++) {
        uint32_t lo = cum[i], hi = cum[i + 1]; if (hi > (1u << pb)) hi = 1u << pb;
        for (uint32_t k = lo; k < hi; k++) slot2sym[k] = (uint8_t)i;
    }
}

static inline uint64_t rans_take(uint64_t x, const uint32_t *F, const uint32_t *cum, uint8_t s, int pb) {
    uint64_t mask = (1ull << pb) - 1; /* ref :292, :483 */
    return (uint64_t)F[s] * (x >> pb) + (x & mask) - cum[s];
}

/* ref: libxpng.c:429-493 */
uint64_t xo_block_v2_decode(const uint8_t *in, uint8_t *out, uint64_t *n_out) {
    uint32_t w0 = ld32(in), type = w0 >> 24;
    if (type == 0) { *n_out = 0; return 4; }
    uint64_t csz = w0 & 0xFFFFFF; uint32_t w1 = ld32(in + 4), n = w1 & 0xFFFFFF, v2 = w1 >> 24;
    *n_out = n;
    if (type == 1) { memset(out, (int)v2, n); return csz; }
    if (type == 2) {
        bitr_t b = { in + 8, in + csz, 0 };
        for (uint32_t i = 0; i < n; i++) out[i] = (uint8_t)br_get(&b, v2);
        return csz;
    }
    unsigned N = v2 + 2; uint32_t w2 = ld32(in + 8); int pb = (int)(w2 >> 24);
    const uint8_t *tab = in + 8 + 4 * (uint64_t)(w2 & 0xFFFFFF), *lo = in + 12;
    uint32_t F[258], cum[259]; static __thread uint8_t slot2sym[1 << 15];
    bitr_t b = { tab, in + csz, 0 };
    get_freq_table(&b, F, N, pb, type == 4);
    build_slot_table(slot2sym, cum, F, N, pb);
    const uint8_t *rp = tab - 16; uint64_t x0 = ld64(rp), x1 = ld64(rp + 8), mask = (1ull << pb) - 1;
    int64_t i = (int64_t)n;
    if (n & 1) { /* ref :471-476 */
        uint8_t s = slot2sym[x0 & mask]; out[--i] = s; x0 = rans_take(x0, F, cum, s, pb);
        if (x0 < RANS_L) { if (rp > lo) rp -= 4; x0 = (x0 << 32) | ld32(rp); }
    }
    for (i -= 2; i >= 0; i -= 2) { /* ref :478-489: fills the output from the end */
        uint8_t s1 = slot2sym[x1 & mask], s0 = slot2sym[x0 & mask];
        out[i + 1] = s1; out[i] = s0;
        x1 = rans_take(x1, F, cum, s1, pb); x0 = rans_take(x0, F, cum, s0, pb);
        if (x1 < RANS_L) { if (rp > lo) rp -= 4; x1 = (x1 << 32) | ld32(rp); }
        if (x0 < RANS_L) { if (rp > lo) rp -= 4; x0 = (x0 << 32) | ld32(rp); }
    }
    return csz;
}

/* v1 block (ref: libxpng.c:160-260).  The reference grows its output downward in a scratch area;
 * here the block is produced in a temporary and returned front-to-back, which yields the same
 * bytes: [hdr][n][state0][state1][renorm words in ascending symbol order].  The frequency table or
 * the raw symbols go to the tile's shared side bit stream `sb`. Returns block size in bytes. */
static uint64_t block_v1_encode(uint32_t *F, unsigned N, const uint8_t *in, uint64_t n,
                                uint8_t *out, bitw_t *sb, int pb) {
    uint32_t nbit = bitlen(N - 1);
    if (n == 0) { st32(out, 4); return 4; }
    unsigned used = 0; for (unsigned i = 0; i < N; i++) used += F[i] != 0;
    if (used == 1) { st32(out, 8u | (1u << 24)); st32(out + 4, (uint32_t)n | ((uint32_t)in[n - 1] << 24)); return 8; }

    uint32_t cum[257]; encsym_t e[256];
    normalise_freqs(F, cum, N, n, pb);
    build_encsyms(e, F, cum, N, pb);

    /* Backward pass (ref :215-245).  Words are emitted in descending symbol order and stored at
     * descending addresses; collect them in emission order, then reverse. */
    uint32_t *tmp = (uint32_t *)malloc(4 * (n + 8)); uint64_t nw = 0;
    uint64_t x0 = RANS_L, x1 = RANS_L; int64_t i = (int64_t)n;
    if (n & 1) { x0 = rans_put(x0, e + in[--i]); } /* ref :218-225: no renorm test */
    for (i -= 2; i >= 0; i -= 2) {
        const encsym_t *s1 = e + in[i + 1], *s0 = e + in[i];
        if (x1 >= rans_limit(s1, pb)) { tmp[nw++] = (uint32_t)x1; x1 >>= 32; }
        if (x0 >= rans_limit(s0, pb)) { tmp[nw++] = (uint32_t)x0; x0 >>= 32; }
        x1 = rans_put(x1, s1); x0 = rans_put(x0, s0);
    }
    uint64_t payload = 16 + 4 * nw; /* states + words (ref :250: *_res - res before the header) */
    uint32_t tab_bits = (N - used) + used * ((uint32_t)pb + 1);
    int sparse = tab_bits < N * (uint32_t)pb;
    tr_put(XO_D_V1_TABLE, (uint32_t)sparse, tab_bits, N * (uint32_t)pb, used, N);
    if (!sparse) tab_bits = N * (uint32_t)pb;
    tr_put(XO_D_V1_BLOCK, tab_bits + 8 * payload < (uint64_t)nbit * n, tab_bits + 8 * payload, (uint64_t)nbit * n, n, N);

    if (tab_bits + 8 * payload >= (uint64_t)nbit * n) { /* ref :250-254 raw symbols into sb */
        for (uint64_t k = 0; k < n; k++) bw_put(sb, nbit, in[k]);
        st32(out, 8u | (2u << 24)); st32(out + 4, (uint32_t)n);
        free(tmp); return 8;
    }
    put_freq_table(sb, F, N, pb, sparse, 1); /* ref :256-257 */
    uint64_t size = 8 + payload;
    st32(out, (uint32_t)size | ((uint32_t)(3 + sparse) << 24)); st32(out + 4, (uint32_t)n);
    st64(out + 8, x0); st64(out + 16, x1);
    for (uint64_t k = 0; k < nw; k++) st32(out + 24 + 4 * k, tmp[nw - 1 - k]);
    free(tmp);
    return size;
}

/* ref: libxpng.c:262-301.  Returns bytes consumed from `in`. */
static uint64_t block_v1_decode(const uint8_t *in, unsigned N, uint8_t *out, uint64_t *n_out,
                                bitr_t *sb, int pb) {
    uint32_t nbit = bitlen(N - 1), w0 = ld32(in), type = w0 >> 24; uint64_t size = w0 & 0xFFFFFF;
    *n_out = 0;
    if (type == 0 || type > 4) return size;
    uint32_t w1 = ld32(in + 4);
    if (type == 1) { *n_out = w1 & 0xFFFFFF; memset(out, (int)(w1 >> 24), w1 & 0xFFFFFF); return size; }
    if (type == 2) { *n_out = w1; for (uint32_t i = 0; i < w1; i++) out[i] = (uint8_t)br_get(sb, nbit); return size; }
    uint32_t n = w1, F[256], cum[257]; static __thread uint8_t slot2sym[1 << 15];
    *n_out = n;
    get_freq_table(sb, F, N, pb, type == 4);
    build_slot_table(slot2sym, cum, F, N, pb);
    const uint8_t *end = in + size, *rp = in + 24;
    if (rp > end) return size;
    uint64_t x0 = ld64(in + 8), x1 = ld64(in + 16), mask = (1ull << pb) - 1, i = 0;
    for (; i + 1 < n; i += 2) { /* ref :287-298: forward */
        uint8_t s0 = slot2sym[x0 & mask], s1 = slot2sym[x1 & mask];
        out[i] = s0; out[i + 1] = s1;
        x0 = rans_take(x0, F, cum, s0, pb); x1 = rans_take(x1, F, cum, s1, pb);
        if (x0 < RANS_L) { x0 = (x0 << 32) | (rp + 4 <= end ? ld32(rp) : 0); if (rp < end) rp += 4; }
        if (x1 < RANS_L) { x1 = (x1 << 32) | (rp + 4 <= end ? ld32(rp) : 0); if (rp < end) rp += 4; }
    }
    if (n & 1) out[i] = slot2sym[x0 & mask];
    return size;
}

/* ------------------------------------------------------------------ mode 1 (App. A.3) */

typedef struct { int r[3]; } res3_t;

/* Residual of the pixel at (x,y) of a tile before zig-zag (ref :510-513, :41-44).
 * Row 0 -> left, column 0 -> up, interior -> avg2/grad3 with optional green subtraction. */
static inline res3_t residual_at(const uint8_t *p, uint64_t x, uint64_t y, int64_t bpr, int pxsz,
                                 int Y, int G) {
    res3_t o;
    for (int c = 0; c < 3; c++) {
        int pr;
        if (y == 0) pr = p[c - pxsz];
        else if (x == 0) pr = p[c - bpr];
        else pr = Y ? pred_grad3(p[c - pxsz], p[c - bpr], p[c - bpr - pxsz]) : pred_avg2(p[c - pxsz], p[c - bpr]);
        o.r[c] = p[c] - pr;
    }
    if (G && x > 0 && y > 0) { o.r[0] -= o.r[1]; o.r[2] -= o.r[1]; }
    return o;
}

/* ref: libxpng.c:497-532 + the first-pixel write of :547 */
uint64_t xo_m1_front(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr_, int pxsz,
                     unsigned pr, uint8_t *streams, uint32_t lens[10], uint32_t F[512],
                     uint32_t *kwords) {
    const int64_t bpr = (int64_t)bpr_; const int Y = (pr >> 1) & 1, G = pr & 1;
    uint64_t npx = w * h;
    uint8_t *seq = (uint8_t *)malloc(npx ? npx : 1), *ctx = (uint8_t *)malloc(npx ? npx : 1);
    uint8_t *alpha = streams + npx; uint64_t m = 0, na = 0; uint32_t prev = 0;
    memset(F, 0, 512 * sizeof(uint32_t));
    bitw_t k = { 0, 0, (uint8_t *)kwords };
    for (int c = 0; c < pxsz; c++) bw_put(&k, 8, tile[c]);
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++) {
        const uint8_t *p = tile + y * bpr_ + x * (uint64_t)pxsz;
        if (pxsz == 4) { /* ref :497-502: alpha predicted from the left, column 0 from above */
            int ap = (x == 0) ? p[3 - bpr] : p[3 - 4];
            uint32_t v = zz8(p[3] - ap);
            alpha[na++] = (uint8_t)v; F[256 + v]++;
            if (p[3] == 0) continue;
        }
        res3_t d = residual_at(p, x, y, bpr, pxsz, Y, G);
        uint32_t u0 = zz8(d.r[0]), u1 = zz8(d.r[1]), u2 = zz8(d.r[2]), nl = bitlen(u0 | u1 | u2);
        F[prev * 16 + nl]++; ctx[m] = (uint8_t)prev; seq[m++] = (uint8_t)nl; prev = nl;
        if (nl) bw_put(&k, 3 * nl, (u0 << (2 * nl)) | (u1 << nl) | u2);
    }
    bw_end(&k);
    /* stable 9-way split of seq by context (ref :504: *cx[pl]++ = nl) */
    uint64_t off[10]; off[0] = 0;
    for (int c = 0; c < 9; c++) { uint32_t s = 0; for (int v = 0; v < 16; v++) s += F[c * 16 + v]; lens[c] = s; off[c + 1] = off[c] + s; }
    lens[9] = (uint32_t)na;
    uint64_t cur[9]; memcpy(cur, off, sizeof cur);
    for (uint64_t i = 0; i < m; i++) streams[cur[ctx[i]]++] = seq[i];
    if (pxsz == 4 && off[9] != npx) memmove(streams + off[9], alpha, na);
    free(seq); free(ctx);
    return (uint64_t)(k.out - (uint8_t *)kwords) / 4;
}

/* ref: libxpng.c:534-571 */
uint64_t xo_encode_tile_m1(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr, int pxsz,
                           uint8_t *out) {
    uint64_t npx = w * h;
    unsigned pr = xo_select_predictor(tile, w, h, bpr, pxsz);
    uint8_t *streams = (uint8_t *)malloc(2 * npx + 16); uint32_t lens[10], F[512];
    uint64_t kw = xo_m1_front(tile, w, h, bpr, pxsz, pr, streams, lens, F, (uint32_t *)(out + 8));
    st32(out + 4, (uint32_t)(4 + 4 * kw));
    uint8_t *f = out + 8 + 4 * kw; const uint8_t *s = streams;
    for (int c = 0; c < 9; c++) { tr_stream = (uint32_t)c; f += xo_block_v2_encode(F + c * 16, 9, s, lens[c], f, 12); s += lens[c]; }
    tr_stream = 9;
    if (pxsz == 4) f += xo_block_v2_encode(F + 256, 256, s, lens[9], f, 15);
    free(streams);
    uint64_t raw = npx * (uint64_t)pxsz + 4, coded = (uint64_t)(f - out);
    tr_stream = 0;
    tr_put(XO_D_T1_TILE, coded < raw, coded, raw, pr, npx);
    if (coded < raw) { st32(out, (1u << 28) + (pr << 24) + (uint32_t)coded); return coded; }
    st32(out, (uint32_t)raw); /* ref :566-567 raw tile */
    for (uint64_t y = 0; y < h; y++) memcpy(out + 4 + y * w * pxsz, tile + y * bpr, w * pxsz);
    return raw;
}

/* ref: libxpng.c:796-863 */
static void decode_tile_m1(const uint8_t *f, uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr_, int pxsz) {
    const int64_t bpr = (int64_t)bpr_; uint64_t npx = w * h; uint32_t m = f[3];
    if (!m) { for (uint64_t y = 0; y < h; y++) memcpy(tile + y * bpr_, f + 4 + y * w * pxsz, w * pxsz); return; }
    const int Y = (m >> 1) & 1, G = m & 1;
    uint32_t bsz = ld32(f + 4);
    bitr_t k = { f + 8, f + 4 + bsz, 0 };
    for (int c = 0; c < pxsz; c++) tile[c] = (uint8_t)br_get(&k, 8);
    uint8_t *sym = (uint8_t *)malloc(2 * npx + 16), *cx[10]; const uint8_t *blk = f + 4 + bsz;
    cx[0] = sym;
    for (int c = 0; c < 9; c++) { uint64_t n; blk += xo_block_v2_decode(blk, cx[c], &n); cx[c + 1] = cx[c] + n; }
    if (pxsz == 4) { uint64_t n; xo_block_v2_decode(blk, cx[9], &n); }
    uint32_t nl = 0;
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++) {
        uint8_t *p = tile + y * bpr_ + x * (uint64_t)pxsz;
        if (pxsz == 4) {
            int ap = (x == 0) ? p[3 - bpr] : p[3 - 4];
            p[3] = (uint8_t)(unzz(*cx[9]++) + ap);
            if (p[3] == 0) { p[0] = p[1] = p[2] = 0; continue; }
        }
        nl = *cx[nl]++;
        int r[3] = { 0, 0, 0 };
        if (nl) {
            uint32_t v = br_get(&k, 3 * nl), mk = (1u << nl) - 1;
            r[0] = unzz(v >> (2 * nl)); r[1] = unzz((v >> nl) & mk); r[2] = unzz(v & mk);
        }
        if (G && x > 0 && y > 0) { r[0] += r[1]; r[2] += r[1]; }
        for (int c = 0; c < 3; c++) {
            int pd;
            if (y == 0) pd = p[c - pxsz];
            else if (x == 0) pd = p[c - bpr];
            else pd = Y ? pred_grad3(p[c - pxsz], p[c - bpr], p[c - bpr - pxsz]) : pred_avg2(p[c - pxsz], p[c - bpr]);
            p[c] = (uint8_t)(r[c] + pd);
        }
    }
    free(sym);
}

/* ------------------------------------------------------------------ mode 2 (App. A.5) */

static const unsigned M2_ALPHABET[9] = { 9, 8, 64, 8, 16, 32, 64, 128, 256 }; /* ref :669 */

/* ref: libxpng.c:628-643 */
static int tile_is_single_colour(const uint8_t *t, uint64_t w, uint64_t h, uint64_t bpr, int pxsz) {
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = 0; x < w; x++)
        if (memcmp(t, t + y * bpr + x * (uint64_t)pxsz, (size_t)pxsz)) return 0;
    return 1;
}

/* ref: libxpng.c:583-626.  Returns blob size, or 0 if the tile is not grey. */
static uint64_t encode_tile_grey(const uint8_t *t, uint64_t w, uint64_t h, uint64_t bpr_, uint8_t *out) {
    const int64_t bpr = (int64_t)bpr_; uint64_t npx = w * h, n = npx - 1;
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = 0; x < w; x++) {
        const uint8_t *p = t + y * bpr_ + 3 * x; if (p[0] != p[1] || p[1] != p[2]) return 0;
    }
    uint8_t *st = (uint8_t *)malloc(4 * npx + 4); uint32_t (*F)[256] = calloc(4, sizeof *F); uint64_t k = 0;
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++, k++) {
        const uint8_t *p = t + y * bpr_ + 3 * x; int v = p[0], c[4];
        if (y == 0) c[0] = c[1] = c[2] = c[3] = v - p[-3];
        else if (x == 0) c[0] = c[1] = c[2] = c[3] = v - p[-bpr];
        else {
            c[0] = v - p[-3]; c[1] = v - p[-bpr];
            c[2] = v - pred_avg2(p[-3], p[-bpr]); c[3] = v - pred_grad3(p[-3], p[-bpr], p[-bpr - 3]);
        }
        for (int i = 0; i < 4; i++) { uint32_t u = zz8(c[i]); st[i * npx + k] = (uint8_t)u; F[i][u]++; }
    }
    uint8_t *bits[4], *blk[4]; uint64_t bsz[4], rsz[4]; unsigned best = 0;
    for (unsigned i = 0; i < 4; i++) {
        bits[i] = (uint8_t *)malloc(2 * npx + 4096); blk[i] = (uint8_t *)malloc(4 * npx + 4096);
        bitw_t b = { t[0], 8, bits[i] + 4 };
        tr_stream = i;
        rsz[i] = block_v1_encode(F[i], 256, st + i * npx, n, blk[i], &b, 15);
        bw_end(&b); bsz[i] = (uint64_t)(b.out - bits[i]); st32(bits[i], (uint32_t)bsz[i]);
        if (bsz[i] + rsz[i] < bsz[best] + rsz[best]) best = i; /* ref :612 strict <, ties -> lowest */
    }
    tr_stream = 0;
    tr_put(XO_D_GREY_PICK, best, bsz[0] + rsz[0], bsz[1] + rsz[1], bsz[2] + rsz[2], bsz[3] + rsz[3]);
    tr_put(XO_D_GREY_PLANE, bsz[best] + rsz[best] < npx, bsz[best] + rsz[best], npx, best, npx);
    uint64_t size;
    if (bsz[best] + rsz[best] >= npx) { /* ref :615-619 raw grey plane */
        size = npx + 4; st32(out, (uint32_t)size + (5u << 27));
        for (uint64_t y = 0, q = 4; y < h; y++) for (uint64_t x = 0; x < w; x++) out[q++] = t[y * bpr_ + 3 * x];
    } else {
        size = bsz[best] + rsz[best] + 4;
        st32(out, (uint32_t)size + (2u << 28) + (best << 24));
        memcpy(out + 4, bits[best], bsz[best]); memcpy(out + 4 + bsz[best], blk[best], rsz[best]);
    }
    for (unsigned i = 0; i < 4; i++) { free(bits[i]); free(blk[i]); }
    free(st); free(F);
    return size;
}

/* ref: libxpng.c:645-686 (+ :33-44 ENC macros) */
uint64_t xo_encode_tile_m2(const uint8_t *t, uint64_t w, uint64_t h, uint64_t bpr_, uint8_t *out) {
    const int64_t bpr = (int64_t)bpr_; uint64_t npx = w * h;
    if (tile_is_single_colour(t, w, h, bpr_, 3)) { /* ref :637-640 */
        st32(out, (255u << 24) | 8); out[4] = t[0]; out[5] = t[1]; out[6] = t[2]; out[7] = 0; return 8;
    }
    uint64_t g = encode_tile_grey(t, w, h, bpr_, out);
    if (g) return g;

    unsigned pr = xo_select_predictor(t, w, h, bpr_, 3); const int Y = (pr >> 1) & 1, G = pr & 1;
    uint32_t (*F)[256] = calloc(9, sizeof *F);
    uint8_t *cx[9], *sv[9]; uint64_t ncx[9] = { 0 }, nsv[9] = { 0 };
    for (int i = 0; i < 9; i++) { cx[i] = (uint8_t *)malloc(npx + 1); sv[i] = (uint8_t *)malloc(3 * npx + 3); }
    uint32_t prev = 0;
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++) {
        const uint8_t *p = t + y * bpr_ + 3 * x;
        res3_t d = residual_at(p, x, y, bpr, 3, Y, G);
        uint32_t u0 = zz8(d.r[0]), u1 = zz8(d.r[1]), u2 = zz8(d.r[2]), nl = bitlen(u0 | u1 | u2);
        F[0][prev * 16 + nl]++; cx[prev][ncx[prev]++] = (uint8_t)nl; prev = nl;
        if (nl == 1) { uint32_t v = (u0 << 2) | (u1 << 1) | u2; sv[1][nsv[1]++] = (uint8_t)v; F[1][v]++; }
        else if (nl == 2) { uint32_t v = (u0 << 4) | (u1 << 2) | u2; sv[2][nsv[2]++] = (uint8_t)v; F[2][v]++; }
        else if (nl) { sv[nl][nsv[nl]++] = (uint8_t)u0; sv[nl][nsv[nl]++] = (uint8_t)u1; sv[nl][nsv[nl]++] = (uint8_t)u2;
                       F[nl][u0]++; F[nl][u1]++; F[nl][u2]++; }
    }
    uint8_t *bits = (uint8_t *)malloc(4 * npx + 65536), *blocks = (uint8_t *)malloc(6 * npx + 65536), *bp = blocks;
    bitw_t b = { ((uint32_t)t[0] << 16) | ((uint32_t)t[1] << 8) | t[2], 24, bits + 4 }; /* ref :659-660 */
    for (int i = 0; i < 9; i++) { tr_stream = (uint32_t)i; bp += block_v1_encode(F[0] + i * 16, 9, cx[i], ncx[i], bp, &b, 14); }
    for (int i = 1; i < 9; i++) { tr_stream = 8 + (uint32_t)i; bp += block_v1_encode(F[i], M2_ALPHABET[i], sv[i], nsv[i], bp, &b, 14); }
    bw_end(&b);
    uint64_t bsz = (uint64_t)(b.out - bits), rsz = (uint64_t)(bp - blocks), size; st32(bits, (uint32_t)bsz);
    tr_stream = 0;
    tr_put(XO_D_T2_TILE, bsz + rsz < npx * 3, bsz + rsz, npx * 3, pr, npx);
    if (bsz + rsz >= npx * 3) { /* ref :675-677 raw tile */
        size = npx * 3 + 4; st32(out, (uint32_t)size);
        for (uint64_t y = 0; y < h; y++) memcpy(out + 4 + y * w * 3, t + y * bpr_, w * 3);
    } else {
        size = bsz + rsz + 4; st32(out, (uint32_t)size + (1u << 28) + (pr << 24));
        memcpy(out + 4, bits, bsz); memcpy(out + 4 + bsz, blocks, rsz);
    }
    for (int i = 0; i < 9; i++) { free(cx[i]); free(sv[i]); }
    free(bits); free(blocks); free(F);
    return size;
}

/* ref: libxpng.c:868-961 */
static void decode_tile_m2(const uint8_t *f, uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr_) {
    const int64_t bpr = (int64_t)bpr_; uint64_t npx = w * h; uint32_t m = f[3];
    if (!m) { for (uint64_t y = 0; y < h; y++) memcpy(tile + y * bpr_, f + 4 + y * w * 3, w * 3); return; }
    if (m == 255) { /* ref :916-927 */
        for (uint64_t y = 0; y < h; y++) for (uint64_t x = 0; x < w; x++) memcpy(tile + y * bpr_ + 3 * x, f + 4, 3);
        return;
    }
    if ((m >> 4) == 2) { /* grey, ref :868-899 */
        if (m & 8) { for (uint64_t y = 0, q = 4; y < h; y++) for (uint64_t x = 0; x < w; x++) { uint8_t *p = tile + y * bpr_ + 3 * x; p[0] = p[1] = p[2] = f[q++]; } return; }
        uint32_t bsz = ld32(f + 4), pm = m & 3; bitr_t b = { f + 8, f + 4 + bsz, 0 };
        tile[0] = tile[1] = tile[2] = (uint8_t)br_get(&b, 8);
        uint8_t *st = (uint8_t *)malloc(npx + 1); uint64_t n, k = 0;
        block_v1_decode(f + 4 + bsz, 256, st, &n, &b, 15);
        for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++) {
            uint8_t *p = tile + y * bpr_ + 3 * x; int v = unzz(st[k++]), pd;
            if (y == 0) pd = p[-3];
            else if (x == 0) pd = p[-bpr];
            else switch (pm) {
                case 0: pd = p[-3]; break;
                case 1: pd = p[-bpr]; break;
                case 2: pd = pred_avg2(p[-3], p[-bpr]); break;
                default: pd = pred_grad3(p[-3], p[-bpr], p[-bpr - 3]);
            }
            p[0] = p[1] = p[2] = (uint8_t)(v + pd);
        }
        free(st); return;
    }
    const int Y = (m >> 1) & 1, G = m & 1;
    uint32_t bsz = ld32(f + 4); bitr_t b = { f + 8, f + 4 + bsz, 0 };
    for (int c = 0; c < 3; c++) tile[c] = (uint8_t)br_get(&b, 8);
    const uint8_t *blk = f + 4 + bsz; uint8_t *cx[9], *sv[9], *cxb[9], *svb[9]; uint64_t n;
    for (int i = 0; i < 9; i++) { cxb[i] = cx[i] = (uint8_t *)malloc(npx + 1); blk += block_v1_decode(blk, 9, cx[i], &n, &b, 14); }
    svb[0] = sv[0] = NULL;
    for (int i = 1; i < 9; i++) { svb[i] = sv[i] = (uint8_t *)malloc(3 * npx + 3); blk += block_v1_decode(blk, M2_ALPHABET[i], sv[i], &n, &b, 14); }
    uint32_t nl = 0;
    for (uint64_t y = 0; y < h; y++) for (uint64_t x = (y == 0); x < w; x++) {
        uint8_t *p = tile + y * bpr_ + 3 * x; int r[3] = { 0, 0, 0 };
        nl = *cx[nl]++;
        if (nl == 1) { uint32_t v = *sv[1]++; r[0] = unzz(v >> 2); r[1] = unzz((v >> 1) & 1); r[2] = unzz(v & 1); }
        else if (nl == 2) { uint32_t v = *sv[2]++; r[0] = unzz(v >> 4); r[1] = unzz((v >> 2) & 3); r[2] = unzz(v & 3); }
        else if (nl) { r[0] = unzz(sv[nl][0]); r[1] = unzz(sv[nl][1]); r[2] = unzz(sv[nl][2]); sv[nl] += 3; }
        if (G && x > 0 && y > 0) { r[0] += r[1]; r[2] += r[1]; }
        for (int c = 0; c < 3; c++) {
            int pd;
            if (y == 0) pd = p[c - 3];
            else if (x == 0) pd = p[c - bpr];
            else pd = Y ? pred_grad3(p[c - 3], p[c - bpr], p[c - bpr - 3]) : pred_avg2(p[c - 3], p[c - bpr]);
            p[c] = (uint8_t)(r[c] + pd);
        }
    }
    for (int i = 0; i < 9; i++) { free(cxb[i]); free(svb[i]); }
}

/* ------------------------------------------------------------------ file level (App. A.1) */

/* ref: libxpng.c:723-789 */
uint64_t xo_encode(int mode, const uint8_t *px_in, uint64_t w, uint64_t h, int A, uint8_t *out) {
    if (!w || !h || w > (1u << 24) || h > (1u << 24) || !px_in || !(mode == 1 || mode == 2 || mode == 7)) return 0;
    A = A ? 1 : 0;
    uint64_t s; uint8_t *px = (uint8_t *)malloc(w * h * (3 + (uint64_t)A));
    A = xo_normalize(px_in, w, h, A, px, &s);
    const int pxsz = 3 + A; const uint64_t bpr = w * (uint64_t)pxsz;
    if (s <= 4) mode = 7;
    uint32_t h0 = (uint32_t)(w - 1) | ((uint32_t)mode << 24), h1 = (uint32_t)(h - 1) | ((uint32_t)A << 24);
    uint64_t size = 0;
    if (mode == 7) goto stored;
    if (mode == 2 && tile_is_single_colour(px, w, h, bpr, pxsz)) { /* ref :741-753 */
        st32(out, h0); st32(out + 4, h1 | (2u << 24)); memcpy(out + 8, px, (size_t)pxsz);
        free(px); return 8 + (uint64_t)pxsz;
    }
    if (A && mode == 2) { mode = 1; h0 = (uint32_t)(w - 1) | (1u << 24); } /* ref :755 */
    if (A && (w < 4 || h < 4)) { free(px); return 0; } /* reference crashes here (SURVEY App. C.1) */
    {
        uint64_t N = xo_tile_grid(w, h, pxsz, NULL, 0);
        xo_tile_t *tl = (xo_tile_t *)malloc(N * sizeof *tl); xo_tile_grid(w, h, pxsz, tl, N);
        uint8_t *blob = (uint8_t *)malloc(8 * 700 * 700 + 65536); uint64_t total = 0; int overflow = 0;
        for (uint64_t i = 0; i < N; i++) {
            const uint8_t *tp = px + tl[i].y * bpr + tl[i].x * (uint64_t)pxsz;
            tr_tile = (uint32_t)i; tr_stream = 0;
            uint64_t bs = mode == 1 ? xo_encode_tile_m1(tp, tl[i].w, tl[i].h, bpr, pxsz, blob)
                                    : xo_encode_tile_m2(tp, tl[i].w, tl[i].h, bpr, blob);
            if (!overflow && total + bs < s) memcpy(out + 8 + total, blob, bs); else overflow = 1;
            total += bs;
        }
        free(blob); free(tl);
        tr_tile = (uint32_t)N; tr_stream = 0;
        tr_put(XO_D_FILE, total < s, total, s, N, (uint64_t)mode);
        if (total >= s) { mode = 7; h0 = (uint32_t)(w - 1) | (7u << 24); goto stored; } /* ref :771-777 */
        st32(out, h0); st32(out + 4, h1); size = 8 + total;
        free(px); return size;
    }
stored:
    st32(out, (uint32_t)(w - 1) | (7u << 24)); st32(out + 4, h1); memcpy(out + 8, px, s);
    free(px); return 8 + s;
}

/* ref: libxpng.c:969-973 */
int xo_peek(const uint8_t *file, uint64_t n, uint64_t *w, uint64_t *h, int *A, int *mode) {
    if (n < 8) return 1;
    uint32_t h0 = ld32(file), h1 = ld32(file + 4);
    *w = (h0 & 0xFFFFFF) + 1; *h = (h1 & 0xFFFFFF) + 1; *A = (h1 >> 24) & 1; *mode = (int)(h0 >> 24);
    return !(*mode == 1 || *mode == 2 || *mode == 7);
}

/* ref: libxpng.c:963-997 */
int xo_decode(const uint8_t *file, uint64_t n, uint8_t *px) {
    uint64_t w, h; int A, mode;
    if (xo_peek(file, n, &w, &h, &A, &mode)) return 1;
    const int pxsz = 3 + A; const uint64_t bpr = w * (uint64_t)pxsz, s = bpr * h;
    if (mode == 7) { if (n < 8 + s) return 1; memcpy(px, file + 8, s); return 0; }
    if (n == 11 + (uint64_t)A && (file[7] & 2)) { /* ref :976-980 */
        for (uint64_t i = 0; i < w * h; i++) memcpy(px + i * pxsz, file + 8, (size_t)pxsz);
        return 0;
    }
    uint64_t N = xo_tile_grid(w, h, pxsz, NULL, 0), off = 8;
    xo_tile_t *tl = (xo_tile_t *)malloc(N * sizeof *tl); xo_tile_grid(w, h, pxsz, tl, N);
    for (uint64_t i = 0; i < N; i++) {
        if (off + 4 > n) { free(tl); return 1; }
        const uint8_t *f = file + off; uint8_t *tp = px + tl[i].y * bpr + tl[i].x * (uint64_t)pxsz;
        if (mode == 1) decode_tile_m1(f, tp, tl[i].w, tl[i].h, bpr, pxsz);
        else decode_tile_m2(f, tp, tl[i].w, tl[i].h, bpr);
        off += ld32(f) & 0xFFFFFF;
    }
    free(tl);
    return 0;
}

/* ------------------------------------------------------------------ YCoCg-R side experiment */

/* ref: Tell_Me_Why/YCoCg-R.c:22 and :31 */
void xo_ycocg_r_fwd(int R, int G, int B, int *Y, int *Co, int *Cg) {
    int co = R - B, t = B + (co >> 1), cg = G - t;
    *Co = co; *Cg = cg; *Y = t + (cg >> 1);
}
void xo_ycocg_r_inv(int Y, int Co, int Cg, int *R, int *G, int *B) {
    int t = Y - (Cg >> 1), g = Cg + t, b = t - (Co >> 1);
    *G = g; *B = b; *R = b + Co;
}
