/*
 * xpng_b200.h — batch / in-memory C ABI of the B200-native xPNG codec.
 *
 * The reference (alantudyk/xPNG) exposes only a file-at-a-time API (xpng.h:12-20, re-declared in
 * include/xpng.h and implemented on top of this interface).  This header adds what a GPU needs to
 * be measured and sharded: N images in, N `.xpng` byte strings out (and back), with the pixels and
 * the compressed bytes in HOST or DEVICE memory.  Plain C types only; no CUDA or torch types.
 *
 * Reference interfaces replaced:
 *   xpngb_encode  <->  xpng_store_T   (libxpng.c:723-789) minus the fopen/fwrite
 *   xpngb_decode  <->  xpng_load_T    (libxpng.c:963-997) minus the f_read/malloc
 *   xpngb_peek    <->  header parse   (libxpng.c:969-973)
 * All functions return 0 on success and non-zero on failure (the reference's _Bool convention).
 */
#ifndef XPNG_B200_H
#define XPNG_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct xpngb_ctx xpngb_ctx;

/* One image of a batch.  `offset` is the byte offset of its pixels (interleaved 8-bit RGB or RGBA,
 * row-major, w*h*(3+A) bytes) inside the pixel buffer; it must be a multiple of 16. */
typedef struct xpngb_image {
    uint64_t w, h;
    uint64_t offset;
    uint32_t A;        /* 1 = RGBA */
    uint32_t mode;     /* out (encode): level actually written (1, 2, 7); out (decode): level found */
} xpngb_image;

/* Create / destroy a codec context bound to CUDA device `device`.  Fails (non-zero) when no usable
 * CUDA device exists: there is no CPU fallback. */
int xpngb_create(xpngb_ctx **ctx, int device);
void xpngb_destroy(xpngb_ctx *ctx);
const char *xpngb_last_error(const xpngb_ctx *ctx);

/* Upper bound of the output bytes xpngb_encode needs for these images (16-byte padded files). */
uint64_t xpngb_encode_bound(const xpngb_image *imgs, uint32_t n);

/* Encode n images at `level` (1, 2 or 7).
 *   pixels / pixels_on_device : base of the pixel buffer (host or device memory), `pixels_size` bytes
 *   out / out_on_device       : receives the .xpng files, file i at out_offsets[i], out_sizes[i] bytes
 * imgs[i].A and imgs[i].mode are updated to what the file header says (alpha may be stripped by the
 * normalisation of libxpng.c:688-721; a level may fall back to 7). */
int xpngb_encode(xpngb_ctx *ctx, int level, xpngb_image *imgs, uint32_t n,
                 const void *pixels, uint64_t pixels_size, int pixels_on_device,
                 void *out, uint64_t out_cap, int out_on_device,
                 uint64_t *out_offsets, uint64_t *out_sizes);

/* Read w, h, A, mode from the first 8 bytes of a .xpng file held in host memory. */
int xpngb_peek(const void *file, uint64_t size, xpngb_image *img);

/* Decode n files.  imgs[i] must carry w, h, A (from xpngb_peek) and `offset` = where image i's
 * pixels go inside `pixels` (multiple of 16).  files / pixels may live on host or device. */
int xpngb_decode(xpngb_ctx *ctx, xpngb_image *imgs, uint32_t n,
                 const void *files, uint64_t files_size, int files_on_device,
                 const uint64_t *file_offsets, const uint64_t *file_sizes,
                 void *pixels, uint64_t pixels_cap, int pixels_on_device);

/* ---- Region decode.  A coded (level 1 / 2) image is cut into independent tiles of at most 666 x 666 pixels, so a
 * rectangle of it can be decoded by decoding only the tiles it touches. */
typedef struct xpngb_rect { uint64_t x, y, w, h; } xpngb_rect;   /* pixels; x, y = top-left corner */

/* Tiles that a region decode of `r` inside a w x h coded (level 1 / 2) image decodes; 0 when r is empty or not inside
 * the image (or w, h exceed the format's 2^24).  *cover (may be NULL) receives their union: a rectangle of whole tiles,
 * in image pixels.  Host only. */
uint32_t xpngb_region_tiles(uint64_t w, uint64_t h, const xpngb_rect *r, xpngb_rect *cover);

/* xpngb_decode of rectangle rects[i] of file i only.  Crop i is written as rects[i].h packed rows of
 * rects[i].w * (3 + A) bytes at pixels + imgs[i].offset (a multiple of 16).  imgs[i] in/out exactly as for xpngb_decode
 * (w, h, A from xpngb_peek: the FULL image; mode out).  The same file may appear in several entries.  Entries with
 * equal (file_offsets[i], file_sizes[i]) share one decode, here and in every call below that takes rectangles, ops,
 * sizes or a tensor format: the tiles of the bounding box of their rectangles' tiles are decoded once into a scratch
 * window, and every entry of the group is cropped (turned, resized, ...) from there.  Equal bytes at different offsets
 * are decoded once per offset.  The output bytes are those of decoding each entry on its own; xpngb_last_tiles counts
 * the shared tiles once.
 * Every entry is checked before anything is decoded: an empty rectangle, one not inside its image, a crop past
 * pixels_cap or a misaligned offset fails the call (xpngb_last_error names the entry), as do the header checks of
 * xpngb_decode.  Corrupt data in a decoded tile fails the call as in a full decode.  Of the tiles a rectangle does not
 * touch only the 4-byte size words up to the last touched tile row are read: their payload is not checked.
 * Level-7 (stored) rectangles are copied straight out of the file.  With host buffers the whole files still cross PCIe. */
int xpngb_decode_region(xpngb_ctx *ctx, xpngb_image *imgs, const xpngb_rect *rects, uint32_t n,
                        const void *files, uint64_t files_size, int files_on_device,
                        const uint64_t *file_offsets, const uint64_t *file_sizes,
                        void *pixels, uint64_t pixels_cap, int pixels_on_device);

/* Traversal-order operations of the exchange scheme (Mirroring_and_Rotating/tool.c:3-127; op codes in the order of
 * its option table, tool.c:133).  TL and TR are empty functions in the reference and therefore plain copies. */
enum { XPNGB_OP_R90 = 0, XPNGB_OP_R270 = 1, XPNGB_OP_MV = 2, XPNGB_OP_MH = 3, XPNGB_OP_MVH = 4, XPNGB_OP_TL = 5, XPNGB_OP_TR = 6 };

/* Apply `op` to n pixmaps: image i is read at src + imgs[i].offset and written at dst + imgs[i].offset (same byte
 * count, so the same offsets serve both buffers; src and dst must not overlap).  imgs[i].w and .h are swapped for the
 * quarter turns.  Replaces op_mv/op_mh/op_mvh/op_r90/op_r270 (tool.c:3-119). */
int xpngb_transform(xpngb_ctx *ctx, int op, xpngb_image *imgs, uint32_t n,
                    const void *src, uint64_t size, int src_on_device, void *dst, int dst_on_device);

/* xpngb_encode of the images as `op` would leave them — the "change the traversal order instead of transforming the
 * pixmap" idea of Mirroring_and_Rotating/README.md:1-4: the files are byte-identical to `tool --op` followed by
 * `xpng -level`, the caller's pixels are not touched, imgs[i].w/.h report the encoded orientation. */
int xpngb_encode_oriented(xpngb_ctx *ctx, int level, int op, xpngb_image *imgs, uint32_t n,
                          const void *pixels, uint64_t pixels_size, int pixels_on_device,
                          void *out, uint64_t out_cap, int out_on_device,
                          uint64_t *out_offsets, uint64_t *out_sizes);

/* xpngb_decode (rects == NULL) or xpngb_decode_region (rects != NULL), with entry i written as `tool --<ops[i]>` would
 * leave what those calls write for it: one op per entry, in the same call.
 *   ops     : non-NULL, ops[i] one of XPNGB_OP_*.  An unknown op fails the call before anything is launched
 *             (xpngb_last_error names the entry).  XPNGB_OP_TL and XPNGB_OP_TR are copies in the reference: those
 *             entries are byte-identical to the unoriented call.
 *   rects   : in the file's coordinates, as stored; the op is applied to the crop afterwards.  NULL: whole images.
 *   output  : packed rows at pixels + imgs[i].offset, the same byte count as the unoriented call.  For R90 and R270 the
 *             width and height are swapped: rects[i].w rows of rects[i].h pixels (whole image: w rows of h pixels).
 *   imgs[i] : in/out exactly as for xpngb_decode (the file's w, h, A; mode out).  Not swapped, so the array can be reused.
 * Every other check is that of xpngb_decode / xpngb_decode_region.  Turned entries are decoded into a scratch window and
 * then written turned (stored level-7 entries are read straight from the file), so they cost one more read and write of
 * their pixels in device memory; with host buffers nothing more crosses PCIe.
 * Files written by xpngb_encode_oriented(op) are restored by the inverse op: XPNGB_OP_R270 for XPNGB_OP_R90,
 * XPNGB_OP_R90 for XPNGB_OP_R270, and `op` itself for every other op. */
int xpngb_decode_oriented(xpngb_ctx *ctx, const int *ops, xpngb_image *imgs, const xpngb_rect *rects, uint32_t n,
                          const void *files, uint64_t files_size, int files_on_device,
                          const uint64_t *file_offsets, const uint64_t *file_sizes,
                          void *pixels, uint64_t pixels_cap, int pixels_on_device);

/* ---- Resized decode: each image or crop resampled to a requested size in the same call, for fixed-size batches. */
typedef struct xpngb_size { uint32_t w, h; } xpngb_size;

/* Entry i is orient(ops[i], resize(crop_i, sizes[i].w, sizes[i].h)), where crop_i is rects[i] in the stored file's
 * coordinates (rects == NULL: the whole image), and ops == NULL means no op (otherwise as for xpngb_decode_oriented).
 *   resize  : byte-identical to Pillow's Image.resize((w, h), Image.BILINEAR) of the crop (8-bit path: horizontal pass
 *             first, rounded to bytes, then vertical; 22-bit fixed-point weights).  Alpha is resampled as a fourth
 *             independent channel, NOT premultiplied: it equals PIL's resize of each channel as an "L" image, and differs
 *             from PIL's own RGBA resize, which premultiplies.
 *   output  : sizes[i].h packed rows of sizes[i].w * (3 + A) bytes at pixels + imgs[i].offset (a multiple of 16).  The op
 *             is applied after the resize, so R90 and R270 write sizes[i].w rows of sizes[i].h pixels.
 *   imgs[i] : in/out exactly as for xpngb_decode (the file's w, h, A; mode out).
 * Every entry is checked before anything is decoded, and the error (xpngb_last_error) names the entry: every check of
 * xpngb_decode_region and xpngb_decode_oriented, sizes == NULL, a zero w or h or one above 2^24, an output past
 * pixels_cap, and a resampled crop side above 2^23 pixels (the 32-bit accumulator of the passes is exact up to there).
 * An entry whose size equals its crop is byte-identical to xpngb_decode_oriented / xpngb_decode_region and takes their
 * path.  Resized entries are decoded into a scratch window (stored level-7 entries are read straight from the file) and
 * resampled in device memory: with host buffers only the resized outputs cross PCIe back. */
int xpngb_decode_resized(xpngb_ctx *ctx, const int *ops, xpngb_image *imgs, const xpngb_rect *rects,
                         const xpngb_size *sizes, uint32_t n,
                         const void *files, uint64_t files_size, int files_on_device,
                         const uint64_t *file_offsets, const uint64_t *file_sizes,
                         void *pixels, uint64_t pixels_cap, int pixels_on_device);

/* ---- Tensor decode: each entry written as the normalised tensor a network takes, in the same call. */
enum { XPNGB_DT_U8 = 0, XPNGB_DT_F32 = 1, XPNGB_DT_F16 = 2, XPNGB_DT_BF16 = 3 };
enum { XPNGB_CHW = 0, XPNGB_HWC = 1 };
enum { XPNGB_SCALE_DIV = 0, XPNGB_SCALE_MUL = 1 };   /* torchvision v1 to_tensor / v2 ToDtype(scale=True) */
typedef struct xpngb_tensor {
    uint32_t dtype, layout, scale;
    uint32_t channels;          /* 3: RGB only (alpha dropped); 0: as stored, 3 + A */
    float mean[4], std[4];      /* per output channel; only the first C are used */
} xpngb_tensor;

/* Entry i's pixels P_i are what xpngb_decode_resized writes for it (sizes == NULL: no resize, as xpngb_decode_oriented /
 * xpngb_decode_region; rects == NULL: whole images; ops == NULL: no op).  They are written as a tensor of C channels:
 * C = 3 when fmt->channels == 3 (alpha dropped, as PIL's convert("RGB")), else 3 + A.  H and W are the output's dimensions
 * after the op.  For each byte b of channel c, every float operation in IEEE float32, round-to-nearest-even, each rounded
 * on its own:
 *   XPNGB_DT_U8   : b (scale, mean and std unused)
 *   XPNGB_DT_F32  : v = b / 255.0f (XPNGB_SCALE_DIV) or v = b * (float)(1.0 / 255) (XPNGB_SCALE_MUL); y = (v - mean[c]) / std[c]
 *   XPNGB_DT_F16, XPNGB_DT_BF16 : that float32 y rounded to nearest-even into the 16-bit type
 *   layout        : XPNGB_CHW puts element (c, y, x) at c*H*W + y*W + x; XPNGB_HWC at (y*W + x)*C + c.
 * DIV + F32 is torchvision's F.normalize(F.to_tensor(pil), mean, std); MUL + F32 is v2.Normalize(mean, std) after
 * v2.ToDtype(torch.float32, scale=True); F16 / BF16 are those passed through .to(dtype); U8 + CHW is F.pil_to_tensor.
 * mean 0, std 1 gives either pipeline without Normalize, bit for bit.
 *   out     : entry i's C*H*W elements at out + imgs[i].offset (a multiple of 16).  A (N, 3, 224, 224) float32 batch uses
 *             offset i * 602112.
 *   imgs[i] : in/out exactly as for xpngb_decode (the file's w, h, A; mode out).
 * Every check runs before anything is decoded, and xpngb_last_error names the entry or the field: every check of
 * xpngb_decode_resized (without sizes: of xpngb_decode_oriented / xpngb_decode_region), fmt == NULL, an unknown dtype,
 * layout or scale, channels other than 0 or 3, for a float dtype a std[c] that is zero or not finite or a mean[c] that is
 * not finite for c < C (all 4 channels when channels == 0), and an output past out_cap.
 * Every entry goes through a scratch window (stored level-7 entries are read straight from their files), and resized
 * entries through a scratch copy of their resized pixels, before one launch per chunk writes the tensors.  Device output
 * is the intended use: with host output a float32 tensor is 4 times the uint8 bytes over PCIe (float16 / bfloat16: 2). */
int xpngb_decode_tensor(xpngb_ctx *ctx, const xpngb_tensor *fmt, const int *ops, xpngb_image *imgs,
                        const xpngb_rect *rects, const xpngb_size *sizes, uint32_t n,
                        const void *files, uint64_t files_size, int files_on_device,
                        const uint64_t *file_offsets, const uint64_t *file_sizes,
                        void *out, uint64_t out_cap, int out_on_device);

/* ---- Resampled decode: Pillow's five convolution filters per entry, and a window of the resized image.
 * Entry i is orient(ops[i], window_i(resize_f(crop_i, sizes[i]))): crop_i is rects[i] (NULL: whole images); resize_f is
 * Pillow's Image.resize(sizes[i], filters[i]) of the crop, byte-identical (Resample.c, 8-bit path), every channel on its
 * own (alpha not premultiplied); window_i keeps windows[i] = (x, y, w, h) in the coordinates of the sizes[i] image (NULL:
 * all of it); the op comes last.  fmt == NULL writes uint8 pixels as xpngb_decode_resized, else a tensor as
 * xpngb_decode_tensor.  filters == NULL and windows == NULL give exactly what xpngb_decode_resized / xpngb_decode_tensor
 * give.  An entry writes windows[i].w * windows[i].h pixels (or tensor elements).  Only the tiles under the support of its
 * window are decoded.  Every check of those calls runs before anything is launched, plus, naming the entry: an unknown
 * filter (NEAREST included: Pillow does not resize with it by convolution), sizes == NULL, an empty window or one not
 * inside sizes[i], and a resampled crop side above the filter's accumulator limit (2^23 box, bilinear and hamming; 2^22
 * bicubic; 2^21 lanczos). */
enum { XPNGB_LANCZOS = 1, XPNGB_BILINEAR = 2, XPNGB_BICUBIC = 3, XPNGB_BOX = 4, XPNGB_HAMMING = 5 };   /* PIL.Image.Resampling */
int xpngb_decode_resampled(xpngb_ctx *ctx, const xpngb_tensor *fmt /* NULL: uint8 pixels, as xpngb_decode_resized */,
                           const int *filters /* NULL: all bilinear */, const int *ops, xpngb_image *imgs,
                           const xpngb_rect *rects, const xpngb_size *sizes /* required */,
                           const xpngb_rect *windows /* NULL: whole resized image */, uint32_t n,
                           const void *files, uint64_t files_size, int files_on_device,
                           const uint64_t *file_offsets, const uint64_t *file_sizes,
                           void *out, uint64_t out_cap, int out_on_device);
/* Diagnostics of the weight tables: Pillow's number of weights per output coordinate of an in -> out axis (0 for in == out
 * or an unknown filter), and the device's tables for output coordinates first .. first + count - 1: xmin_n gets 2 * count
 * int32 (xmin, n), k count * ksize int32 22-bit weights, zero past each window. */
uint32_t xpngb_resize_ksize(int filter, uint32_t in, uint32_t out);
int xpngb_resize_coeffs(xpngb_ctx *ctx, int filter, uint32_t in, uint32_t out, uint32_t first, uint32_t count,
                        int32_t *xmin_n, int32_t *k);

/* ---- Colour decode: torchvision's ColorJitter and RandomGrayscale per entry, byte-identical to their PIL path.
 * Entry i is tensor(gray_i(jitter_i(orient(ops[i], window_i(resize_f(crop_i)))))): what xpngb_decode_resampled writes for it
 * (sizes == NULL: what xpngb_decode_tensor / xpngb_decode_oriented write without a resize; filters and windows then must be
 * NULL), with colors[i]'s steps applied to its 8-bit pixels before the tensor conversion (fmt == NULL: uint8 output).
 *   jitter_i : the steps k = order[0], order[1], ... whose bit k of `on` is set, each mapping bytes to bytes as Pillow does
 *              (every float / double operation rounded on its own):
 *     L(p)        = (19595 R + 38470 G + 7471 B + 0x8000) >> 16, Pillow's L24 luma;
 *     BRIGHTNESS, CONTRAST, SATURATION: Image.blend(d, p, f) per colour channel: a = (float)factor,
 *                 t = (float)d + a * (float)(p - d), out = t <= 0 ? 0 : t >= 255 ? 255 : (int)t, with d = 0 (brightness),
 *                 L(p) (saturation) or m = (int)((double)S / N + 0.5) (contrast), S the sum of L over the entry's N output
 *                 pixels as they stand at that step (ImageStat's mean).  Alpha is unchanged;
 *     HUE         : Pillow's rgb2hsv, H += (uint8_t)(int32_t)(factor * 255.0) mod 256, hsv2rgb (Convert.c).  On RGBA the
 *                 alpha becomes 255: torchvision's adjust_hue converts through HSV, which has no alpha, and that quirk is kept.
 *   gray_i   : gray == 1 sets R = G = B = L(p) after the jitter (RandomGrayscale(num_output_channels=3)).
 * The steps are per pixel and contrast's mean does not depend on pixel order, so the op may come before or after them: the
 * library applies them to the entry's pixels as written.  colors == NULL, or entries with on == 0 and gray == 0, give exactly
 * what xpngb_decode_resampled / xpngb_decode_tensor / xpngb_decode_oriented give.  Every check of those calls runs before
 * anything is launched, plus, naming the entry: an order that is not a permutation of 0..3, a bit of `on` above 3, gray other
 * than 0 or 1, a brightness, contrast or saturation factor that is negative or not finite (also as a float), a hue factor
 * outside [-0.5, 0.5] or NaN, and gray on an entry whose output keeps alpha (uint8 output or channels == 0 of an RGBA file:
 * torchvision's RandomGrayscale refuses 4 channels).  Coloured tensor entries are first written as uint8 pixels into scratch
 * (resized entries already are); one launch per chunk sums the luma of the entries with contrast on, and one applies the chain. */
enum { XPNGB_CJ_BRIGHTNESS = 0, XPNGB_CJ_CONTRAST = 1, XPNGB_CJ_SATURATION = 2, XPNGB_CJ_HUE = 3 };   /* ColorJitter's fn_idx */
typedef struct xpngb_color {
    uint8_t  order[4];   /* the steps in the order applied: a permutation of 0..3, as ColorJitter.get_params' fn_idx */
    uint32_t on;         /* bit k: step k applied (a None factor of get_params: bit clear) */
    uint32_t gray;       /* 1: RandomGrayscale after the jitter */
    double   factor[4];  /* brightness, contrast, saturation: finite, >= 0; hue: in [-0.5, 0.5] */
} xpngb_color;
int xpngb_decode_color(xpngb_ctx *ctx, const xpngb_tensor *fmt /* NULL: uint8 pixels */, const int *filters, const int *ops,
                       xpngb_image *imgs, const xpngb_rect *rects, const xpngb_size *sizes /* NULL: no resize */,
                       const xpngb_rect *windows, const xpngb_color *colors /* NULL: none */, uint32_t n,
                       const void *files, uint64_t files_size, int files_on_device,
                       const uint64_t *file_offsets, const uint64_t *file_sizes,
                       void *out, uint64_t out_cap, int out_on_device);

/* ---- Blurred and solarized decode: Pillow's ImageFilter.GaussianBlur and ImageOps.solarize per entry, byte-identical to Pillow.
 * Entry i is tensor(solarize_i(blur_i(gray_i(jitter_i(orient(ops[i], window_i(resize_f(crop_i)))))))): what xpngb_decode_color
 * writes for it, with blurs[i] applied to its 8-bit pixels after the colour step and before the tensor conversion.  Both act
 * on the entry's output image: the blur's x axis is the output's, and its edges are the output's edges.
 *   blur_i     : img.filter(ImageFilter.GaussianBlur((radius[0], radius[1]))), Pillow's BoxBlur.c.  Per axis, with the radius
 *                narrowed to float and every operation below in float:
 *                  sigma2 = r * r / 3, L = (float)sqrt(sigma2 * 12 + 1), l = floor((L - 1) / 2),
 *                  a = (2l + 1) * (l * (l + 1) - 3 * sigma2) / (6 * (sigma2 - (l + 1) * (l + 1))), fr = l + a,
 *                  ri = (int)fr, ww = (uint32)(16777216.f / (fr * 2 + 1)), fw = (2^24 - (2 ri + 1) * ww) / 2 (uint32).
 *                One pass along a line of one channel, edges clamped to the nearest pixel, in uint32:
 *                  acc = sum of p[clamp(x + k)], k = -ri .. ri; bulk = acc * ww + (p[clamp(x - ri - 1)] + p[clamp(x + ri + 1)]) * fw;
 *                  out = (bulk + 2^23) >> 24, a byte that the next pass reads.
 *                Three passes along x with radius[0], then three along y with radius[1]; an axis whose float radius is 0 is
 *                skipped.  Every channel is blurred on its own, alpha included (no premultiplication).
 *   solarize_i : solarize == 1: every byte v < threshold is kept, every other becomes 255 - v (ImageOps.solarize(img,
 *                threshold); 128 is its default).  All bytes of the output are treated: the call refuses it where alpha is kept.
 * blurs == NULL, or entries with radius {0, 0} and solarize == 0, give exactly what xpngb_decode_color gives.  Every check of
 * xpngb_decode_color runs before anything is launched, plus, naming the entry: a radius that is negative or not finite, a
 * radius above XPNGB_BLUR_RADIUS_MAX as a float, solarize other than 0 or 1, a NaN threshold, and solarize on an entry whose
 * output keeps alpha (uint8 output or channels == 0 of an RGBA file: ImageOps.solarize refuses RGBA).
 * XPNGB_BLUR_RADIUS_MAX = 2^23 is the accumulator bound: up to it (2 ri + 1) * ww <= 2^24, so no uint32 above can wrap
 * (acc * ww + far * fw + 2^23 <= 255 * 2^24 + 2^23); at the next float, 8388609, ri = 2^23, ww = 1 and fw wraps.  The box
 * pass walks each line with a running sum, so its cost does not depend on the radius.  Blurred or solarized tensor entries
 * are staged as uint8 pixels in scratch, as coloured ones are; tensor entries turned by r90 or r270 sit there un-turned and
 * get the passes along y first with radius[0], then along x with radius[1], which equals blurring the turned image. */
#define XPNGB_BLUR_RADIUS_MAX 8388608.0
typedef struct xpngb_blur {
    double   radius[2];   /* ImageFilter.GaussianBlur's (x, y) radius; {0, 0}: no blur */
    uint32_t solarize;    /* 1: ImageOps.solarize after the blur */
    double   threshold;   /* bytes v < threshold are kept, the others become 255 - v */
} xpngb_blur;
int xpngb_decode_blur(xpngb_ctx *ctx, const xpngb_tensor *fmt /* NULL: uint8 pixels */, const int *filters, const int *ops,
                      xpngb_image *imgs, const xpngb_rect *rects, const xpngb_size *sizes /* NULL: no resize */,
                      const xpngb_rect *windows, const xpngb_color *colors /* NULL: none */,
                      const xpngb_blur *blurs /* NULL: none */, uint32_t n,
                      const void *files, uint64_t files_size, int files_on_device,
                      const uint64_t *file_offsets, const uint64_t *file_sizes,
                      void *out, uint64_t out_cap, int out_on_device);
/* Diagnostics: the host's box radius, ww and fw for one axis, as Pillow's _gaussian_blur_radius + ImagingHorizontalBoxBlur.
 * Returns 1 (and sets nothing) for a radius the decode refuses: negative, not finite or above XPNGB_BLUR_RADIUS_MAX. */
int xpngb_blur_box(double radius, int32_t *ri, uint32_t *ww, uint32_t *fw);

/* ---- Auto-augmented decode: torchvision's AutoAugment, RandAugment and TrivialAugmentWide ops (_apply_op on the PIL path)
 * per entry, byte-identical to Pillow.  Entry i is
 *   tensor(solarize_i(blur_i(gray_i(jitter_i(augment_i(orient(ops[i], window_i(resize_f(crop_i)))))))))
 * : what xpngb_decode_blur writes for it, with augs[i]'s program run on its 8-bit RGB image right after the op, where
 * torchvision's ClassificationPresetTrain runs the policy (after RandomResizedCrop and the flip).  Every step acts on the
 * output image: its axes, its size and its edges.  A program is up to XPNGB_AUG_STEPS_MAX steps, run in order; each step is
 * one of the Pillow operations _apply_op ends in, with its parameters as Pillow receives them (xpng_b200.codec.augment_params
 * builds them from (op_name, magnitude) as torchvision does):
 *   AFFINE       img.transform(img.size, Image.AFFINE, data, resample, fillcolor=fill): ShearX/Y, TranslateX/Y and the
 *                Rotate angles without a fast path.  data: the inverse matrix; arg: resample, NEAREST 0, BILINEAR 2 or
 *                BICUBIC 3 (PIL numbering); fill: the RGB fill bytes of the pixels whose source is outside.  NEAREST follows
 *                Pillow's three code paths (scale, 16.16 fixed point, running double sums), BILINEAR / BICUBIC its generic
 *                transform with its filters, all in double with every operation rounded on its own.
 *   TRANSPOSE    Image.rotate's fast paths: arg is XPNGB_OP_MVH (180), XPNGB_OP_R270 (ROTATE_90, square images only) or
 *                XPNGB_OP_R90 (ROTATE_270, square only); any op code is accepted, a quarter turn only on a square output.
 *   BRIGHTNESS, COLOR, CONTRAST   ImageEnhance.*(img).enhance(value): xpngb_decode_color's blends (value narrowed to float).
 *   SHARPNESS    ImageEnhance.Sharpness(img).enhance(value): Image.blend(img.filter(SMOOTH), img, value); SMOOTH is
 *                1 1 1 / 1 5 1 / 1 1 1 over 13, rounded, border rows and columns copied, images with a side below 3 copied.
 *   POSTERIZE    ImageOps.posterize(img, arg): arg bits 0 .. 8 kept.
 *   SOLARIZE     ImageOps.solarize(img, value): bytes v < value kept, others 255 - v.
 *   AUTOCONTRAST, EQUALIZE, INVERT   ImageOps.autocontrast(img), ImageOps.equalize(img), ImageOps.invert(img): per RGB
 *                channel, from the entry's histograms (a single-valued channel, or equalize's step 0, is left unchanged).
 * augs == NULL, or entries with nsteps == 0, give exactly what xpngb_decode_blur gives.  An RGBA file written with
 * channels == 3 is augmented as its RGB image (img.convert("RGB")).  Every check of xpngb_decode_blur runs before anything
 * is launched, plus, naming the entry: nsteps above XPNGB_AUG_STEPS_MAX, an unknown kind, a resample other than 0, 2 or 3,
 * a matrix coefficient that is not finite or is 2^64 or more in magnitude (Pillow's running sums could overflow), a
 * TRANSPOSE arg that is not an op code or turns a non-square output a quarter, a negative or non-finite factor, posterize
 * bits above 8, a NaN threshold, and any step on an entry whose output keeps alpha (uint8 output or channels == 0 of an RGBA
 * file: Pillow's ImageOps refuse RGBA and torchvision documents these transforms for RGB).
 * Warps read one buffer and write another: uint8 entries ping-pong between their output and the lane's scratch and end at
 * their output; tensor entries are staged before the op as coloured ones are and map their warps through the op. */
#define XPNGB_AUG_STEPS_MAX 8
enum { XPNGB_AUG_AFFINE = 0, XPNGB_AUG_TRANSPOSE = 1, XPNGB_AUG_BRIGHTNESS = 2, XPNGB_AUG_COLOR = 3, XPNGB_AUG_CONTRAST = 4,
       XPNGB_AUG_SHARPNESS = 5, XPNGB_AUG_POSTERIZE = 6, XPNGB_AUG_SOLARIZE = 7, XPNGB_AUG_AUTOCONTRAST = 8,
       XPNGB_AUG_EQUALIZE = 9, XPNGB_AUG_INVERT = 10 };
typedef struct xpngb_aug_step {
    double   data[6];   /* AFFINE: the inverse matrix (x_src = data[0] x + data[1] y + data[2], y_src likewise, pixel centres) */
    double   value;     /* BRIGHTNESS .. SHARPNESS: the factor; SOLARIZE: the threshold */
    uint32_t kind;      /* XPNGB_AUG_* */
    int32_t  arg;       /* AFFINE: resample; TRANSPOSE: XPNGB_OP_*; POSTERIZE: bits */
    uint8_t  fill[4];   /* AFFINE: fill colour, RGB ([3] unused) */
} xpngb_aug_step;
typedef struct xpngb_augment {
    uint32_t       nsteps;   /* 0: identity */
    xpngb_aug_step step[XPNGB_AUG_STEPS_MAX];
} xpngb_augment;
int xpngb_decode_augment(xpngb_ctx *ctx, const xpngb_tensor *fmt /* NULL: uint8 pixels */, const int *filters, const int *ops,
                         xpngb_image *imgs, const xpngb_rect *rects, const xpngb_size *sizes /* NULL: no resize */,
                         const xpngb_rect *windows, const xpngb_color *colors /* NULL: none */, const xpngb_blur *blurs /* NULL: none */,
                         const xpngb_augment *augs /* NULL: none */, uint32_t n,
                         const void *files, uint64_t files_size, int files_on_device,
                         const uint64_t *file_offsets, const uint64_t *file_sizes,
                         void *out, uint64_t out_cap, int out_on_device);

/* Device time of the kernels of the last encode/decode call on this context, in milliseconds
 * (CUDA events on the context's stream; excludes host<->device copies). */
float xpngb_last_kernel_ms(const xpngb_ctx *ctx);
/* Number of kernel launches issued by the last call. */
uint32_t xpngb_last_launches(const xpngb_ctx *ctx);
/* Number of tiles the last decode call decoded, summed over its chunks.  Stored (level-7) files count 0.  Entries of one
 * call that read the same file (equal offset and size) count the tiles of that file's shared window once. */
uint64_t xpngb_last_tiles(const xpngb_ctx *ctx);
/* Per-kernel timing: while on, every launch is bracketed by CUDA events and synchronised (so the call
 * gets slower); xpngb_profile_report writes "kernel_name total_ms launches\n" lines and returns the
 * length.  Turning profiling on or off clears the table. */
void xpngb_profile(xpngb_ctx *ctx, int on);
uint32_t xpngb_profile_report(const xpngb_ctx *ctx, char *buf, uint32_t cap);
/* The CUDA stream (cudaStream_t as void*) the context launches on. */
void *xpngb_stream(const xpngb_ctx *ctx);

/* ---- Frame batches sharded over the GPUs of one box (host code in C, no NCCL).  The reference's parallel strategy is a
 * tile cursor plus an ordered concatenation (libxpng.c:146-151, :764-769; offset chain :982); frames are independent, so a
 * batch is cut into contiguous shards, every shard is coded on its own device with no data-path exchange, and the one
 * exchange is the table of compressed sizes, from which every participant derives the same offsets. */

/* Frame i of n belongs to shard floor(i * nshards / n); shard k owns [first, first + count). */
void xpngb_shard_range(uint32_t n, uint32_t nshards, uint32_t shard, uint32_t *first, uint32_t *count);
/* Exclusive scan of 16-byte padded sizes: where file i starts when the n files are written back to back. */
void xpngb_packed_offsets(const uint64_t *sizes, uint32_t n, uint64_t *offsets, uint64_t *total);

/* One process: a pool holds one codec context per device and drives each from its own host thread. */
typedef struct xpngb_pool xpngb_pool;
int xpngb_pool_create(xpngb_pool **pool, const int *devices /* NULL: 0..ndev-1 */, uint32_t ndev);
void xpngb_pool_destroy(xpngb_pool *pool);
uint32_t xpngb_pool_size(const xpngb_pool *pool);
xpngb_ctx *xpngb_pool_context(const xpngb_pool *pool, uint32_t k);
const char *xpngb_pool_last_error(const xpngb_pool *pool);
/* xpngb_encode / xpngb_decode of n images in HOST memory, shard k on pool device k.  Encode: `out` must hold
 * xpngb_encode_bound(imgs, n) bytes; shard k writes its files into its own slice of `out`, out_offsets[i] is the
 * position of file i inside `out`, and the files are byte-identical to a one-device call. */
int xpngb_pool_encode(xpngb_pool *pool, int level, xpngb_image *imgs, uint32_t n, const void *pixels, uint64_t pixels_size,
                      void *out, uint64_t out_cap, uint64_t *out_offsets, uint64_t *out_sizes);
int xpngb_pool_decode(xpngb_pool *pool, xpngb_image *imgs, uint32_t n, const void *files, uint64_t files_size,
                      const uint64_t *file_offsets, const uint64_t *file_sizes, void *pixels, uint64_t pixels_cap);

/* One process per device (torchrun-style launch): the size tables of the ranks meet in a POSIX shared-memory segment.
 * `name` must be the same on every rank and unique per job (e.g. the rendezvous port); rank 0 creates the segment. */
typedef struct xpngb_gather xpngb_gather;
int xpngb_gather_open(xpngb_gather **g, const char *name, uint32_t rank, uint32_t world, uint32_t max_items);
/* Collective: rank r passes the sizes of its shard (xpngb_shard_range(n, world, r)); every rank receives all n sizes and
 * the packed offsets derived from them. */
int xpngb_gather_sizes(xpngb_gather *g, uint32_t n, const uint64_t *local_sizes, uint64_t *all_sizes, uint64_t *all_offsets);
void xpngb_gather_close(xpngb_gather *g);

/* Reversible YCoCg-R lifting of n RGB triples on the device (Tell_Me_Why/YCoCg-R.c:22,:31): a side
 * component, NOT part of the .xpng bit stream.  rgb: 3*n bytes; ycc: 3*n int16 (Y, Co, Cg). */
int xpngb_ycocg_forward(xpngb_ctx *ctx, const uint8_t *rgb_host, int16_t *ycc_host, uint64_t n);
int xpngb_ycocg_inverse(xpngb_ctx *ctx, const int16_t *ycc_host, uint8_t *rgb_host, uint64_t n);

#ifdef __cplusplus
}
#endif
#endif
