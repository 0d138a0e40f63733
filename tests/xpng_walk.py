"""Block walker: parse an .xpng file block by block and report which coded-block kinds it holds.

Layout as written by oracle/xpng_oracle.c (xo_encode, xo_encode_tile_m1 / _m2, xo_block_v2_encode, block_v1_encode,
encode_tile_grey).  The walker checks the file's framing while it goes, and raises WalkError where the bytes do not
account for themselves exactly:
- every tile, block and side bit stream ends where its size field says, and the last tile ends the file;
- every rANS frequency table sums to exactly 2^pb;
- the context blocks of a tile hold one symbol per coded pixel after the first (level 2: npx - 1; level 1 RGB:
  npx - 1, RGBA: at most npx - 1), and a level-1 alpha block holds npx - 1.

walk(data, level) returns a set of feature tuples, e.g. ("file", "fallback7"), ("t2", "grey_raw"), ("t1", "pr2"),
("v1val256", "type3"), ("v2ctx", "dominant").  Stream tags: v2ctx / v2alpha (level 1), v1ctx, v1val<N> for the
level-2 value streams of an N-symbol alphabet, v1grey (level-2 grey plane).  Block features:
  type0 .. type4   empty, run, raw bits, rANS with a dense table, rANS with a sparse table
  odd_n            rANS block with an odd symbol count (one state decodes one more symbol)
  tail             rANS block with n % 32 != 0 (the decoders' partial last step)
  words>512        rANS block with more than 512 renormalisation words (refills of the warp decoders' ring)
  w1               a symbol of width 1 in the table
  dominant         a symbol of width >= 2^pb - 4 (the rest of the alphabet shares at most 4 slots)
"""
import struct

import numpy as np

from oracle import pyoracle as po

M2_ALPHABET = (9, 8, 64, 8, 16, 32, 64, 128, 256)   # xpng_oracle.c M2_ALPHABET: contexts, then nl = 1..8


class WalkError(ValueError):
    pass


def _need(cond, what):
    if not cond:
        raise WalkError(what)


def bitlen(v):
    return int(v).bit_length()


class BitReader:
    """MSB-first bits over little-endian 32-bit words (xpng_oracle.c br_get); reading past `end` is an error here."""

    def __init__(self, buf, start, end):
        self.buf, self.start, self.end, self.pos = buf, start, end, 0

    def get(self, c):
        v = 0
        for _ in range(c):
            p = self.start + 4 * (self.pos >> 5)
            _need(p + 4 <= self.end, "bit stream read past its end")
            word = struct.unpack_from("<I", self.buf, p)[0]
            v = (v << 1) | ((word >> (31 - (self.pos & 31))) & 1)
            self.pos += 1
        return v

    def skip(self, c):
        self.pos += c

    def words(self):
        return (self.pos + 31) // 32


def read_table(br, N, pb, sparse):
    """put_freq_table's form: dense pb bits per symbol; sparse 0, or 1 followed by pb bits."""
    F = []
    for _ in range(N):
        F.append(br.get(pb) if (not sparse or br.get(1)) else 0)
    return F


def rans_features(tag, F, pb, n, nwords, out):
    _need(sum(F) == 1 << pb, f"{tag}: frequency table sums to {sum(F)}, not 2^{pb}")
    _need(n >= 2 and sum(1 for f in F if f) >= 2, f"{tag}: rANS block of {n} symbols over {sum(1 for f in F if f)} used")
    if n & 1:
        out.add((tag, "odd_n"))
    if n % 32:
        out.add((tag, "tail"))
    if n < 32:
        out.add((tag, "n<32"))
    if nwords > 512:
        out.add((tag, "words>512"))
    if 1 in F:
        out.add((tag, "w1"))
    if max(F) >= (1 << pb) - 4:
        out.add((tag, "dominant"))


def walk_v2_block(f, q, end, tag, out):
    """One self-delimiting level-1 block at q (xo_block_v2_encode); returns (size, n)."""
    _need(q + 4 <= end, f"{tag}: block header past the tile")
    w0 = struct.unpack_from("<I", f, q)[0]
    typ, csz = w0 >> 24, w0 & 0xFFFFFF
    out.add((tag, f"type{typ}"))
    _need(q + csz <= end, f"{tag}: block of {csz} bytes runs past the tile")
    if typ == 0:
        _need(csz == 4, f"{tag}: empty block of {csz} bytes")
        return 4, 0
    w1 = struct.unpack_from("<I", f, q + 4)[0]
    n = w1 & 0xFFFFFF
    if typ == 1:
        _need(csz == 8 and n > 0, f"{tag}: run block of {csz} bytes, n={n}")
    elif typ == 2:
        nbit = w1 >> 24
        _need(1 <= nbit <= 8 and csz == 8 + 4 * ((n * nbit + 31) // 32), f"{tag}: raw block of {csz} bytes, n={n} x {nbit} bits")
    elif typ in (3, 4):
        N = (w1 >> 24) + 2
        w2 = struct.unpack_from("<I", f, q + 8)[0]
        pb, tab = w2 >> 24, 8 + 4 * (w2 & 0xFFFFFF)
        _need(pb in (12, 15) and 28 <= tab <= csz, f"{tag}: pb={pb}, table at {tab} of {csz}")
        br = BitReader(f, q + tab, q + csz)
        F = read_table(br, N, pb, typ == 4)
        _need(tab + 4 * br.words() == csz, f"{tag}: table ends at {tab + 4 * br.words()}, block at {csz}")
        _need(F[-1] > 0, f"{tag}: alphabet of {N} with an unused top symbol")
        rans_features(tag, F, pb, n, (w2 & 0xFFFFFF) - 5, out)
    else:
        raise WalkError(f"{tag}: block type {typ}")
    return csz, n


def walk_v1_block(f, q, end, N, pb, sb, tag, out):
    """One level-2 block at q (block_v1_encode); its table or raw symbols come next in the side stream sb."""
    _need(q + 4 <= end, f"{tag}: block header past the tile")
    w0 = struct.unpack_from("<I", f, q)[0]
    typ, size = w0 >> 24, w0 & 0xFFFFFF
    out.add((tag, f"type{typ}"))
    _need(q + size <= end, f"{tag}: block of {size} bytes runs past the tile")
    if typ == 0:
        _need(size == 4, f"{tag}: empty block of {size} bytes")
        return 4, 0
    w1 = struct.unpack_from("<I", f, q + 4)[0]
    if typ == 1:
        n = w1 & 0xFFFFFF
        _need(size == 8 and n > 0 and (w1 >> 24) < N, f"{tag}: run block of {size} bytes, word {w1:#x}")
    elif typ == 2:
        n = w1
        _need(size == 8, f"{tag}: raw block of {size} bytes")
        sb.skip(n * bitlen(N - 1))
    elif typ in (3, 4):
        n = w1
        _need(size >= 24 and size % 4 == 0, f"{tag}: rANS block of {size} bytes")
        F = read_table(sb, N, pb, typ == 4)
        rans_features(tag, F, pb, n, (size - 24) // 4, out)
    else:
        raise WalkError(f"{tag}: block type {typ}")
    return size, n


def walk_tile_m1(f, p, size, npx, A, out):
    m = f[p + 3]
    if m == 0:
        _need(size == 4 + npx * (3 + A), f"level-1 raw tile of {size} bytes for {npx} pixels")
        out.add(("t1", "raw"))
        return
    _need(m >> 4 == 1 and (m >> 2) & 1 == A, f"level-1 tile mode {m:#x}")
    out.add(("t1", f"pr{m & 3}"))
    end = p + size
    bsz = struct.unpack_from("<I", f, p + 4)[0]
    _need(bsz >= 4 + 4 * ((8 * (3 + A) + 31) // 32) and bsz % 4 == 0 and p + 4 + bsz <= end, f"level-1 tile: bsz {bsz}")
    q, nctx = p + 4 + bsz, 0
    for j in range(9):
        csz, n = walk_v2_block(f, q, end, "v2ctx", out)
        q, nctx = q + csz, nctx + n
    if A:
        csz, n = walk_v2_block(f, q, end, "v2alpha", out)
        q += csz
        _need(n == npx - 1 and nctx <= npx - 1, f"level-1 RGBA tile: alpha {n}, contexts {nctx}, npx {npx}")
    else:
        _need(nctx == npx - 1, f"level-1 tile: contexts hold {nctx} symbols, npx {npx}")
    _need(q == end, f"level-1 tile: blocks end at {q - p}, tile at {size}")


def walk_tile_m2(f, p, size, npx, out):
    m = f[p + 3]
    end = p + size
    if m == 0:
        _need(size == 4 + 3 * npx, f"level-2 raw tile of {size} bytes for {npx} pixels")
        out.add(("t2", "raw"))
        return
    if m == 255:
        _need(size == 8, f"single-colour tile of {size} bytes")
        out.add(("t2", "single"))
        return
    if m == 0x28:
        _need(size == 4 + npx, f"grey raw tile of {size} bytes for {npx} pixels")
        out.add(("t2", "grey_raw"))
        return
    _need(m >> 4 in (1, 2) and m & 0xC == 0, f"level-2 tile mode {m:#x}")
    grey = m >> 4 == 2
    out.add(("t2", f"grey_pm{m & 3}" if grey else f"pr{m & 3}"))
    bsz = struct.unpack_from("<I", f, p + 4)[0]
    _need(bsz >= 8 and bsz % 4 == 0 and p + 4 + bsz <= end, f"level-2 tile: bsz {bsz}")
    sb = BitReader(f, p + 8, p + 4 + bsz)
    sb.skip(8 if grey else 24)   # the first pixel
    q = p + 4 + bsz
    if grey:
        sz, n = walk_v1_block(f, q, end, 256, 15, sb, "v1grey", out)
        q += sz
        _need(n == npx - 1, f"grey tile: {n} symbols, npx {npx}")
    else:
        nctx = 0
        for j in range(9):
            sz, n = walk_v1_block(f, q, end, 9, 14, sb, "v1ctx", out)
            q, nctx = q + sz, nctx + n
        _need(nctx == npx - 1, f"level-2 tile: contexts hold {nctx} symbols, npx {npx}")
        for N in M2_ALPHABET[1:]:
            sz, n = walk_v1_block(f, q, end, N, 14, sb, f"v1val{N}", out)
            q += sz
    _need(4 * sb.words() == bsz - 4, f"level-2 tile: side stream uses {4 * sb.words()} bytes of {bsz - 4}")
    _need(q == end, f"level-2 tile: blocks end at {q - p}, tile at {size}")


def walk(data, level=None):
    """Feature set of one .xpng file; `level` is the level it was requested at (1, 2 or 7), if known."""
    f = bytes(data)
    _need(len(f) >= 11, "file shorter than a header and a pixel")
    w0, w1 = struct.unpack_from("<II", f, 0)
    W, H, mode, A = (w0 & 0xFFFFFF) + 1, (w1 & 0xFFFFFF) + 1, w0 >> 24, (w1 >> 24) & 1
    pxsz = 3 + A
    out = set()
    if mode == 7:
        _need(len(f) == 8 + W * H * pxsz, f"stored file of {len(f)} bytes for {W}x{H}x{pxsz}")
        out.add(("file", "stored" if level in (None, 7) else "fallback7"))
        return out
    _need(mode in (1, 2), f"file mode {mode}")
    if mode == 2 and (w1 >> 24) & 2:   # xo_encode: one colour for the whole image, 8 + pxsz bytes
        _need(len(f) == 8 + pxsz, f"single-colour file of {len(f)} bytes")
        out.add(("file", "single"))
        return out
    _need((w1 >> 24) & ~1 == 0 and not (mode == 2 and A), f"file header {w0:#x} {w1:#x}")
    out.add(("file", f"m{mode}"))
    p = 8
    for tx, ty, tw, th in po.tile_grid(W, H, pxsz):
        npx = int(tw) * int(th)
        _need(p + 4 <= len(f), "tile header past the file")
        size = struct.unpack_from("<I", f, p)[0] & 0xFFFFFF
        _need(size >= 4 and p + size <= len(f), f"tile of {size} bytes past the file")
        if mode == 1:
            walk_tile_m1(f, p, size, npx, A, out)
        else:
            walk_tile_m2(f, p, size, npx, out)
        p += size
    _need(p == len(f), f"tiles end at {p}, file at {len(f)}")
    return out
