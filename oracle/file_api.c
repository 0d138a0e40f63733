/*
 * file_api.c — the reference's file-at-a-time entry points (xpng.h:17-18) over the CPU oracle.
 *
 * TEST INFRASTRUCTURE ONLY, built into its own library (oracle/libxo_file.so) so that code written
 * against that API (bench.py's file harness) can be checked on a host without a GPU.  T is ignored
 * (single-threaded); 0 = success, 1 = failure; xpng_load_T's pixels are malloc'd (free() them).
 */
#include "xpng_oracle.h"
#include <stdio.h>
#include <stdlib.h>

typedef struct xo_xpng_t { uint8_t *p; uint64_t w, h, s; _Bool A; } xo_xpng_t;   /* layout of xpng_t, xpng.h:10 */

_Bool xpng_store_T(uint64_t T, uint64_t mode, const xo_xpng_t *pm, const char *path);
_Bool xpng_load_T(uint64_t T, const char *path, xo_xpng_t *pm);

/* ref: libxpng.c:723-794 (validation :729-731, file write after the encode) */
_Bool xpng_store_T(uint64_t T, uint64_t mode, const xo_xpng_t *pm, const char *path) {
    (void)T;
    if (!pm || !path || !pm->p || !(mode == 1 || mode == 2 || mode == 7) || !pm->w || !pm->h ||
        pm->w > (1u << 24) || pm->h > (1u << 24) || pm->w * pm->h * (3 + (uint64_t)pm->A) != pm->s) return 1;
    uint8_t *out = (uint8_t *)malloc(8 + pm->s);
    if (!out) return 1;
    const uint64_t n = xo_encode((int)mode, pm->p, pm->w, pm->h, pm->A, out);
    FILE *f = n ? fopen(path, "wb") : NULL;
    _Bool bad = !f || fwrite(out, 1, n, f) != n;
    if (f && fclose(f)) bad = 1;
    free(out);
    return bad;
}

/* ref: libxpng.c:963-1002 */
_Bool xpng_load_T(uint64_t T, const char *path, xo_xpng_t *pm) {
    (void)T;
    if (!path || !pm) return 1;
    FILE *f = fopen(path, "rb");
    if (!f) return 1;
    long n = fseek(f, 0, SEEK_END) ? -1 : ftell(f);
    uint8_t *file = n >= 0 ? (uint8_t *)calloc((size_t)n + 16, 1) : NULL;   /* zero tail: the decoder may read ahead */
    if (!file || fseek(f, 0, SEEK_SET) || fread(file, 1, (size_t)n, f) != (size_t)n) { fclose(f); free(file); return 1; }
    fclose(f);
    uint64_t w, h; int A, mode;
    uint8_t *px = NULL;
    if (xo_peek(file, (uint64_t)n, &w, &h, &A, &mode) || !(px = (uint8_t *)malloc(w * h * (3 + (uint64_t)A))) ||
        xo_decode(file, (uint64_t)n, px)) { free(px); free(file); return 1; }
    free(file);
    pm->p = px; pm->w = w; pm->h = h; pm->s = w * h * (3 + (uint64_t)A); pm->A = A != 0;
    return 0;
}
