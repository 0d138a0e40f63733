/*
 * xpng_oracle.h — CPU restatement of the xPNG encode/decode hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under xpng_b200/ (the product) may include, link or call
 * this.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * use it, as the checker.  It is a from-scratch, single-threaded, in-memory restatement of the
 * algorithm in the reference's libxpng.c; every function cites the reference lines it follows
 * (paths relative to the reference tree).  Parity is PINNED: tests/test_oracle_pin.py compares it
 * byte-for-byte with files produced by the unmodified reference build (oracle/_ref, recipe in
 * oracle/Makefile) and with the committed golden vectors in tests/golden/.
 */
#ifndef XPNG_ORACLE_H
#define XPNG_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct xo_tile_t { uint64_t x, y, w, h; } xo_tile_t;

/* Tile grid of a W x H image with pxsz bytes per pixel (libxpng.c:51-83).  Writes up to cap tiles
 * in row-major tile order; returns the tile count. */
uint64_t xo_tile_grid(uint64_t W, uint64_t H, int pxsz, xo_tile_t *tiles, uint64_t cap);

/* Alpha normalisation (libxpng.c:688-721).  in: w*h*(3+A) bytes.  out: capacity >= input size.
 * Returns the output alpha flag (0/1) and writes the output byte count to *s_out. */
int xo_normalize(const uint8_t *in, uint64_t w, uint64_t h, int A, uint8_t *out, uint64_t *s_out);

/* Predictor/transform selection of one tile (libxpng.c:92-140).  tile points at the tile's first
 * pixel inside an image whose rows are bpr bytes apart. */
unsigned xo_select_predictor(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr, int pxsz);

/* Mode-1 front end of one tile (libxpng.c:497-532): the ten symbol streams (cx0..cx8, alpha)
 * concatenated into `streams` (capacity >= 2*w*h), their lengths, the 512-bin histogram block
 * (F[ctx*16+nl], alpha at F[256+v]) and the residual bit stream k (words, capacity >= w*h + 4).
 * Returns the number of 32-bit words of k. */
uint64_t xo_m1_front(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr, int pxsz,
                     unsigned pr, uint8_t *streams, uint32_t lens[10], uint32_t F[512],
                     uint32_t *kwords);

/* v2 entropy block (libxpng.c:307-427 / :429-493).  F is modified (normalised) as in the
 * reference.  Encode returns the block size in bytes; decode returns the bytes consumed and
 * writes the symbol count to *n_out. */
uint64_t xo_block_v2_encode(uint32_t *F, unsigned nsym, const uint8_t *in, uint64_t n,
                            uint8_t *out, int prob_bits);
uint64_t xo_block_v2_decode(const uint8_t *in, uint8_t *out, uint64_t *n_out);

/* One tile -> tile blob.  `out` must hold 8*w*h + 4096 bytes.  Return blob size (bytes). */
uint64_t xo_encode_tile_m1(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr, int pxsz,
                           uint8_t *out);
uint64_t xo_encode_tile_m2(const uint8_t *tile, uint64_t w, uint64_t h, uint64_t bpr,
                           uint8_t *out);

/* Whole image -> .xpng file bytes (libxpng.c:723-789).  mode in {1,2,7}.  out capacity must be
 * >= 8 + w*h*(3+A).  Returns the file size, or 0 on a validation failure. */
uint64_t xo_encode(int mode, const uint8_t *px, uint64_t w, uint64_t h, int A, uint8_t *out);

/* Header peek (libxpng.c:969-973): returns 0 on success. */
int xo_peek(const uint8_t *file, uint64_t n, uint64_t *w, uint64_t *h, int *A, int *mode);

/* .xpng file bytes -> pixels (libxpng.c:963-997).  px capacity w*h*(3+A).  Returns 0 on success. */
int xo_decode(const uint8_t *file, uint64_t n, uint8_t *px);

/* Decision log: every size comparison the encoder makes, in the order it makes them.  xo_trace(buf, cap) starts a log
 * of this thread into buf (and empties it); xo_trace(NULL, 0) stops it.  xo_trace_len() is the number of decisions
 * made since the start, which may exceed cap (only the first cap are stored).  Logging changes no output.
 *
 *   kind            outcome (1: first side won)        v[0] vs v[1]: the comparison   v[2], v[3]
 *   XO_D_T1_TILE    coded (coded < raw)                coded, raw bytes               predictor, npx
 *   XO_D_FILE       coded (total < s)                  sum of tile sizes, s           tiles, mode
 *   XO_D_T2_TILE    coded (bsz + rsz < 3 npx)          bsz + rsz, 3 npx               predictor, npx
 *   XO_D_GREY_PLANE coded (bsz + rsz < npx)            bsz + rsz of the pick, npx     pick, npx
 *   XO_D_V2_BLOCK   rANS (csz < rawsz)                 csz, rawsz bytes               n, N
 *   XO_D_V2_TABLE   sparse (N + used pb < N pb)        N + used pb, N pb bits         used, N
 *   XO_D_V1_BLOCK   rANS (tab + 8 payload < nbit n)    tab + 8 payload, nbit n bits   n, N
 *   XO_D_V1_TABLE   sparse (tab_sparse < N pb)         (N - used) + used (pb+1), N pb used, N
 *   XO_D_PRED       the index picked                   v[0..3]: the four predictor costs
 *   XO_D_GREY_PICK  the index picked                   v[0..3]: the four grey candidates' bsz + rsz
 *   XO_D_STEAL      the donor                          starved symbol, smallest width >1  symbols of that width, last of them
 * tile is the tile's index in the image (XO_D_FILE: the tile count); stream is the block's stream: level 1 contexts
 * 0..8 and alpha 9, level 2 contexts 0..8 and values 9..16 (nl 1..8), grey candidates 0..3; 0 for tile-level kinds. */
enum { XO_D_T1_TILE = 1, XO_D_FILE, XO_D_T2_TILE, XO_D_GREY_PLANE, XO_D_GREY_PICK, XO_D_V2_BLOCK, XO_D_V2_TABLE,
       XO_D_V1_BLOCK, XO_D_V1_TABLE, XO_D_PRED, XO_D_STEAL };
typedef struct xo_decision_t { uint32_t kind, tile, stream, outcome; uint64_t v[4]; } xo_decision_t;
void xo_trace(xo_decision_t *buf, uint64_t cap);
uint64_t xo_trace_len(void);

/* Reversible YCoCg-R lifting, the side experiment of Tell_Me_Why/YCoCg-R.c:10-34 (NOT on the
 * .xpng path).  Co and Cg are 9-bit signed. */
void xo_ycocg_r_fwd(int R, int G, int B, int *Y, int *Co, int *Cg);
void xo_ycocg_r_inv(int Y, int Co, int Cg, int *R, int *G, int *B);

#ifdef __cplusplus
}
#endif
#endif
