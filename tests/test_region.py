"""Region decode (xpngb_decode_region / Codec.decode_region): a rectangle of each file, decoded from the tiles it touches.

Without a GPU: xpngb_region_tiles against the CPU oracle's own tile grid (oracle/xpng_oracle.c, independent code).
On the GPU: every crop equals the pinned CPU oracle's full decode, cut to the rectangle."""
import ctypes as C
import hashlib
import json
import os
import struct

import numpy as np
import pytest

from conftest import ROOT, make_case, manifest
from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------- tile selection (CPU)

def expected_tiles(w, h, rect):
    """(count, cover) from the oracle's tile grid: the tiles that intersect rect and the bounding box of their union."""
    x, y, rw, rh = rect
    if rw == 0 or rh == 0 or x >= w or y >= h or rw > w - x or rh > h - y:
        return 0, None
    g = po.tile_grid(w, h).astype(np.int64)
    hit = g[(g[:, 0] < x + rw) & (g[:, 0] + g[:, 2] > x) & (g[:, 1] < y + rh) & (g[:, 1] + g[:, 3] > y)]
    x0, y0 = int(hit[:, 0].min()), int(hit[:, 1].min())
    x1, y1 = int((hit[:, 0] + hit[:, 2]).max()), int((hit[:, 1] + hit[:, 3]).max())
    assert (x1 - x0) * (y1 - y0) == int((hit[:, 2] * hit[:, 3]).sum())      # the union of a rows x columns block is a rectangle
    return len(hit), (x0, y0, x1 - x0, y1 - y0)


# one-tile images, strips (w < 444), bands (h < 444), 1080p (first column 588, first row 636), 4K (first two columns 366,
# first two rows 414), 666-wide first tiles (1110 = 2 x 444 + 222), 1 x N and N x 1
SHAPES = [(1, 1), (37, 53), (666, 296), (300, 2000), (2000, 300), (1920, 1080), (3840, 2160), (1110, 1110), (1, 5000), (5000, 1),
          (445, 445), (8192, 8192)]


def selection_cases():
    rng = np.random.default_rng(20261020)
    cases = []
    for w, h in SHAPES:
        g = po.tile_grid(w, h)
        xs, ys = sorted(set(int(v) for v in g[:, 0])), sorted(set(int(v) for v in g[:, 1]))
        cases += [(w, h, (0, 0, w, h)), (w, h, (w - 1, h - 1, 1, 1)), (w, h, (0, 0, 1, 1))]
        # edges on a tile boundary and one pixel either side of it
        for _ in range(8):
            bx, by = xs[int(rng.integers(len(xs)))], ys[int(rng.integers(len(ys)))]
            x0 = min(max(bx + int(rng.integers(-1, 2)), 0), w - 1)
            y0 = min(max(by + int(rng.integers(-1, 2)), 0), h - 1)
            ex, ey = xs[int(rng.integers(len(xs)))] + int(rng.integers(-1, 2)), ys[int(rng.integers(len(ys)))] + int(rng.integers(-1, 2))
            cases.append((w, h, (x0, y0, max(1, min(ex, w) - x0), max(1, min(ey, h) - y0))))
        for _ in range(4):
            x0, y0 = int(rng.integers(w)), int(rng.integers(h))
            cases.append((w, h, (x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1)))))
        # empty, out of range, overflowing: all 0
        cases += [(w, h, (0, 0, 0, h)), (w, h, (0, 0, w, 0)), (w, h, (0, 0, w + 1, h)), (w, h, (0, 0, w, h + 1)), (w, h, (w, 0, 1, 1)),
                  (w, h, (0, h, 1, 1)), (w, h, (2 ** 64 - 1, 0, 2, 1)), (w, h, (1, 0, 2 ** 64 - 1, 1)), (w, h, (0, 2 ** 63, 1, 2 ** 63))]
    return cases


CASES = selection_cases()


def test_selection_case_count():
    assert len(CASES) >= 200


@pytest.mark.parametrize("w,h,rect", CASES, ids=[f"{w}x{h}-{r}" for w, h, r in CASES])
def test_region_tiles_match_oracle_grid(w, h, rect):
    assert xpng_b200.region_tiles(w, h, rect) == expected_tiles(w, h, rect)


def test_region_tiles_whole_image_is_every_tile():
    for w, h in SHAPES:
        n, cover = xpng_b200.region_tiles(w, h, (0, 0, w, h))
        assert n == len(po.tile_grid(w, h)) and cover == (0, 0, w, h)


# ---------------------------------------------------------------------------------------------------- region decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def grid_rects(w, h, rng):
    """1x1 at each corner, random rectangles, rectangles across tile boundaries, exactly one tile, a union of whole tiles
    (decoded in place) and the full image."""
    g = po.tile_grid(w, h).astype(int)
    out = [(0, 0, 1, 1), (w - 1, 0, 1, 1), (0, h - 1, 1, 1), (w - 1, h - 1, 1, 1)]
    for _ in range(3):
        x0, y0 = int(rng.integers(w)), int(rng.integers(h))
        out.append((x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1))))
    for tx, ty, tw, th in g[1:3]:      # across the boundary at the tile's top-left corner
        x0, y0 = max(int(tx) - 7, 0), max(int(ty) - 5, 0)
        out.append((x0, y0, min(19, w - x0), min(13, h - y0)))
    out.append(tuple(int(v) for v in g[int(rng.integers(len(g)))]))
    xs = sorted(set(int(v) for v in g[:, 0]))
    out.append((xs[-1], 0, w - xs[-1], h))    # the last tile column
    out.append((0, 0, w, h))
    return out


def halfflat(h, w, seed):
    d = synth.rgb(h, w, seed)
    d[:, :600] = [10, 200, 30]               # as the `halfflat` manifest entry; the flat part covers the first tile column,
    return d                                 # whose tiles are single-colour tiles at level 2


GENS = {"rgb": synth.rgb, "rgba": synth.rgba, "gray_as_rgb": synth.gray_as_rgb, "noise": synth.noise,
        "flat": lambda h, w, s: np.full((h, w, 3), s % 251, np.uint8), "halfflat": halfflat}


def check(codec, files, rects):
    got = codec.decode_region(files, rects)
    for f, r, g in zip(files, rects, got):
        x, y, w, h = r
        want = po.decode(f)[y: y + h, x: x + w]
        assert g.shape == want.shape and np.array_equal(g, want), r
    return got


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("gen", sorted(GENS))
def test_region_against_oracle(codec, gen, level):
    rng = np.random.default_rng(sorted(GENS).index(gen) * 3 + level)
    h, w = 700, 1000                         # 2 x 2 tiles (350 + 350 rows, 556 + 444 columns)
    f = po.encode(level, GENS[gen](h, w, 41))
    rects = grid_rects(w, h, rng)
    got = check(codec, [f] * len(rects), rects)      # one file, many entries
    assert np.array_equal(got[-1], codec.decode([f])[0])
    for r in rects:                                  # and one entry per call
        check(codec, [f], [r])


@gpu
@pytest.mark.parametrize("name", ("rgba_8192_s2", "rgb_4k_s1"))
def test_region_large_golden(codec, name):
    entry = manifest()["synthetic"][name]
    px = make_case("synthetic", name, entry)
    h, w = px.shape[:2]
    rng = np.random.default_rng(5)
    for lv in (1, 2):
        f = codec.encode(lv, [px])[0]
        assert hashlib.sha256(f).hexdigest() == entry["levels"][str(lv)]["sha256"]
        full = po.decode(f)
        rects = [(w - 256, h - 256, 256, 256), (1000, 1000, 1024, 1024), (int(rng.integers(w - 300)), int(rng.integers(h - 300)), 300, 223),
                 (0, 0, w, h)]
        got = codec.decode_region([f] * len(rects), rects)
        for (x, y, rw, rh), g in zip(rects, got):
            assert np.array_equal(g, full[y: y + rh, x: x + rw]), (name, lv, (x, y, rw, rh))


@gpu
def test_region_mixed_batch(codec):
    imgs = [synth.rgb(900, 1300, 1), synth.rgba(500, 460, 2), synth.gray_as_rgb(300, 520, 3), synth.noise(90, 70, 4),
            np.full((700, 800, 3), 9, np.uint8), synth.rgb(1, 1399, 6), synth.rgb(1823, 1, 5)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7, 1, 2, 2, 1), imgs)]
    rng = np.random.default_rng(9)
    batch, rects = [], []
    for f, im in zip(files, imgs):
        h, w = im.shape[:2]
        for _ in range(3):
            x0, y0 = int(rng.integers(w)), int(rng.integers(h))
            batch.append(f); rects.append((x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1))))
    perm = rng.permutation(len(batch))
    check(codec, [batch[k] for k in perm], [rects[k] for k in perm])


@gpu
def test_region_batch_kernel_family(monkeypatch):
    """The pair decoders, three-tile walk and row-pitched un-predict (selected by batch size), forced on small inputs."""
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(3)
        for lv in (1, 2):
            for im in (synth.rgb(700, 1000, 81), synth.rgba(900, 700, 82), halfflat(700, 1000, 23)):
                h, w = im.shape[:2]
                f = po.encode(lv, im)
                rects = grid_rects(w, h, rng)
                check(cd, [f] * len(rects), rects)
    finally:
        cd.close()


@gpu
def test_region_pipelined_chunks(monkeypatch):
    """64 sintel-like frames with one seeded 224 x 224 crop each, cut into about eight chunks on three lanes (lanes are
    reused within the call), through the batch kernel family."""
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "config3_64.json")))
    frames = synth.sintel_batch(range(1000, 1064))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "3")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "3")      # about 20 MPix of covered tiles in all
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(64)
        rects = [(int(rng.integers(1920 - 224)), int(rng.integers(1080 - 224)), 224, 224) for _ in frames]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for k, f in enumerate(files):
                size, digest = gold[str(1000 + k)][str(lv)]
                assert len(f) == size and hashlib.sha256(f).hexdigest() == digest
            check(cd, files, rects)
    finally:
        cd.close()


@gpu
def test_region_device_resident_buffers(codec):
    import torch
    frames = [synth.rgb(720, 1280, 60), synth.rgba(600, 900, 61), synth.rgb(333, 517, 62)]
    files = [po.encode(lv, f) for lv, f in zip((1, 1, 2), frames)]
    rects = [(100, 37, 600, 500), (0, 444, 900, 156), (17, 3, 1, 300)]
    n = len(files)
    descs = (xpng_b200.codec._Image * n)()
    foffs, fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
    fb, poff = bytearray(), 0
    for i, (f, r) in enumerate(zip(files, rects)):
        foffs[i], fsizes[i] = len(fb), len(f)
        fb += f + b"\0" * (-len(f) % 16)
        descs[i].offset = poff
        poff += (r[2] * r[3] * frames[i].shape[2] + 15) & ~15
    dfiles = torch.from_numpy(np.frombuffer(bytes(fb), np.uint8).copy()).cuda()
    dpx = torch.zeros(poff, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    codec.decode_region_raw(descs, xpng_b200.codec.rects(rects), n, dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dpx.data_ptr(), poff, 1)
    out = dpx.cpu().numpy()
    for i, (f, (x, y, w, h)) in enumerate(zip(files, rects)):
        c = 3 + descs[i].A
        got = out[descs[i].offset: descs[i].offset + w * h * c].reshape(h, w, c)
        assert np.array_equal(got, po.decode(f)[y: y + h, x: x + w])


def scribble_outside(f, w, h, cover, seed):
    """The file with the payload (everything after the 4-byte size word) of every tile outside `cover` replaced by noise."""
    b, rng = bytearray(f), np.random.default_rng(seed)
    off = 8
    cx, cy, cw, ch = cover
    for tx, ty, tw, th in po.tile_grid(w, h).astype(int):       # the tile chain is in raster order of the grid
        size = struct.unpack_from("<I", b, off)[0] & 0xFFFFFF
        inside = cx <= tx < cx + cw and cy <= ty < cy + ch
        if not inside and size > 4:
            b[off + 4: off + size] = rng.integers(0, 256, size - 4, dtype=np.uint8).tobytes()
        off += size
    assert off == len(b)
    return bytes(b)


@gpu
def test_untouched_tiles_are_not_decoded(codec):
    px = synth.rgb(1080, 1920, 77)
    rects = [(600, 700, 224, 224), (588, 636, 444, 444), (1500, 20, 400, 600), (0, 0, 1, 1)]
    for lv in (1, 2):
        f = po.encode(lv, px)
        for r in rects:
            n, cover = xpng_b200.region_tiles(1920, 1080, r)
            assert n < 8
            bad = scribble_outside(f, 1920, 1080, cover, n)
            x, y, w, h = r
            assert np.array_equal(codec.decode_region([bad], [r])[0], px[y: y + h, x: x + w]), (lv, r)


@gpu
def test_region_failures(codec):
    px = synth.rgb(600, 700, 5)
    f = po.encode(1, px)
    bad = bytearray(f); bad[9] ^= 0xFF; bad[10] ^= 0x7F            # first tile's size word
    with pytest.raises(RuntimeError):
        codec.decode_region([bytes(bad)], [(500, 400, 50, 50)])
    for r in [(0, 0, 0, 10), (0, 0, 10, 0), (0, 0, 701, 10), (0, 0, 10, 601), (700, 0, 1, 1), (2 ** 64 - 1, 0, 2, 2),
              (0, 2 ** 64 - 1, 2, 2), (5, 5, 2 ** 64 - 1, 1)]:
        with pytest.raises(RuntimeError, match="entry 1"):
            codec.decode_region([f, f], [(0, 0, 5, 5), r])
    descs = (xpng_b200.codec._Image * 1)()
    fb = np.frombuffer(f + b"\0" * 16, np.uint8)
    foffs, fsizes = (C.c_uint64 * 1)(0), (C.c_uint64 * 1)(len(f))
    rect = xpng_b200.codec.rects([(10, 10, 100, 50)])
    px_out = np.zeros(100 * 50 * 3 + 64, np.uint8)
    with pytest.raises(RuntimeError):            # crop beyond pixels_cap
        codec.decode_region_raw(descs, rect, 1, fb.ctypes.data, len(f), 0, foffs, fsizes, px_out.ctypes.data, 100 * 50 * 3 - 1, 0)
    descs[0].offset = 8
    with pytest.raises(RuntimeError):            # misaligned offset
        codec.decode_region_raw(descs, rect, 1, fb.ctypes.data, len(f), 0, foffs, fsizes, px_out.ctypes.data, len(px_out), 0)
    descs[0].offset = 16
    codec.decode_region_raw(descs, rect, 1, fb.ctypes.data, len(f), 0, foffs, fsizes, px_out.ctypes.data, len(px_out), 0)
    assert np.array_equal(px_out[16: 16 + 15000].reshape(50, 100, 3), px[10:60, 10:110])
