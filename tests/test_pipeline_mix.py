"""Mixed batches across several chunks and lanes, against the CPU oracle.

An encode or decode call cuts its batch into chunks of whole images and runs them on up to XPNGB_PIPE_LANES lanes, each
lane reusing its scratch for its next chunk (cut_chunks, encode_issue, decode_call in csrc/api.cu).  By default a batch is
one chunk below 32 MPix, so here XPNGB_PIPE_MIN_MPIX=1 and XPNGB_CHUNK_MPIX=1 cut a 6 MPix batch into six chunks of
1 MPix on two or three lanes.  The batch of mix() is built so that the chunks hold different content (a level-2 chunk split into its
level-1 and level-2 groups, RGB only, opaque and dirty RGBA, stored and thin images, translucent RGBA only): every lane
runs chunks of different kinds one after the other.  restated_cuts() restates cut_chunks; the batches are checked to
cut into more chunks than lanes, and one call of each kind asserts from the profile that it ran the chunks
the restatement predicts, so that a change of the cuts cannot quietly turn these tests into single-chunk tests.

Without a GPU: the oracle header of every image class, and the restated cuts of the batches.
On the GPU: every file equals po.encode, every decoded image, crop or resize equals the oracle's."""
import ctypes as C
import os
import struct
from functools import lru_cache

import numpy as np
import pytest

from conftest import CORPUS, load_png
from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import _Image, rects, region_tiles, sizes as size_arr
from test_resized_decode import resize_bilinear

gpu = pytest.mark.gpu
MPIX = 1 << 20
KNOBS = {"XPNGB_PIPE_MIN_MPIX": "1", "XPNGB_CHUNK_MPIX": "1"}
GUARD = 4096            # guard bytes after a host output buffer
ALL_OPS = list(po.TOOL_OPS)


def restated_cuts(pxs, lanes, min_px=MPIX, max_px=MPIX):
    """cut_chunks of csrc/api.cu: k chunks of equal pixel share, k = ceil(total / want), want = ceil(total / lanes)
    clamped to [min_px, max_px]; chunk c ends with the image that brings the running count to c / k of the total."""
    n, total = len(pxs), sum(pxs)
    want = min(max(-(-total // lanes), min_px), max_px)
    k = min(max(-(-total // want), 1), n)
    cuts, run, c = [0], 0, 1
    for i in range(n):
        if c >= k:
            break
        run += pxs[i]
        if run * k >= c * total and i + 1 < n:
            cuts.append(i + 1)
            while c < k and run * k >= c * total:
                c += 1
    return cuts + [n]


# ------------------------------------------------------------------------------------------------------------ images

def _opaque(h, w, s):
    return np.ascontiguousarray(np.concatenate([synth.rgb(h, w, s), np.full((h, w, 1), 255, np.uint8)], axis=2))


def _dirty(h, w, s):
    d = synth.rgba(h, w, s)
    d[d[..., 3] == 0] = [9, 8, 7, 0]
    return d


def _translucent(h, w, s):
    """RGB under an alpha that varies and is never 0 or 255 (synth.rgba may leave a small image opaque)."""
    a = (1 + (np.arange(h * w).reshape(h, w, 1) * 7 + s) % 253).astype(np.uint8)
    return np.ascontiguousarray(np.concatenate([synth.rgb(h, w, s), a], axis=2))


def _dirty_clear(h, w, s):
    """Alpha 0 everywhere over non-zero colour: normalised, one colour."""
    d = synth.noise(h, w, s, channels=4)
    d[..., 3] = 0
    return d


GENS = {
    "rgb": synth.rgb, "gray": synth.gray_as_rgb, "noise": synth.noise,
    "rgba": synth.rgba, "translucent": _translucent, "dirty": _dirty, "opaque": _opaque, "dirty_clear": _dirty_clear,
    "flat_rgb": lambda h, w, s: np.full((h, w, 3), 30 + s % 200, np.uint8),
    "flat_rgba": lambda h, w, s: np.full((h, w, 4), 128, np.uint8),
    "clear": lambda h, w, s: np.zeros((h, w, 4), np.uint8),
}

# class -> (generator, shape of the class's example, oracle header (A, mode, single colour) per level; None: rejected)
RGB_HDR = {1: (0, 1, 0), 2: (0, 2, 0), 7: (0, 7, 0)}
RGBA_HDR = {1: (1, 1, 0), 2: (1, 1, 0), 7: (1, 7, 0)}
CLASSES = {
    "rgb": ("rgb", (300, 500), RGB_HDR),
    "gray_as_rgb": ("gray", (200, 300), RGB_HDR),
    "noise": ("noise", (90, 70), {1: (0, 7, 0), 2: (0, 7, 0), 7: (0, 7, 0)}),              # incompressible: stored
    "translucent_rgba": ("rgba", (400, 333), RGBA_HDR),
    "translucent_ramp": ("translucent", (4, 250), RGBA_HDR),
    "dirty_rgba": ("dirty", (300, 260), RGBA_HDR),                                         # colour under alpha 0 zeroed
    "dirty_clear_rgba": ("dirty_clear", (40, 50), {1: (1, 1, 0), 2: (1, 2, 1), 7: (1, 7, 0)}),
    "opaque_rgba": ("opaque", (260, 300), RGB_HDR),                                        # alpha stripped
    "single_rgb": ("flat_rgb", (64, 80), {1: (0, 1, 0), 2: (0, 2, 1), 7: (0, 7, 0)}),
    "single_rgba": ("flat_rgba", (50, 60), {1: (1, 1, 0), 2: (1, 2, 1), 7: (1, 7, 0)}),
    "stored_rgb_1x1": ("flat_rgb", (1, 1), {1: (0, 7, 0), 2: (0, 7, 0), 7: (0, 7, 0)}),    # 4 bytes or less: mode 7
    "stored_rgba_1x1": ("flat_rgba", (1, 1), {1: (1, 7, 0), 2: (1, 7, 0), 7: (1, 7, 0)}),
    "thin_rgb_1xN": ("rgb", (1, 1399), RGB_HDR),
    "thin_rgb_Nx1": ("rgb", (1823, 1), RGB_HDR),
    "thin_opaque_rgba": ("opaque", (50, 2), {1: (0, 1, 0), 2: (0, 7, 0), 7: (0, 7, 0)}),
    "thin_single_rgba": ("flat_rgba", (50, 2), {1: None, 2: (1, 2, 1), 7: (1, 7, 0)}),
    "thin_clear_rgba": ("clear", (50, 3), {1: None, 2: (1, 2, 1), 7: (1, 7, 0)}),
    "thin_translucent_rgba": ("translucent", (50, 2), {1: None, 2: None, 7: (1, 7, 0)}),
    "wide_tile": ("rgb", (37, 1500), RGB_HDR),                                             # one tile 1500 pixels wide
    "largest_tile": ("rgb", (666, 666), RGB_HDR),                                          # one tile of 443 556 pixels
}

# Six groups of exactly 1 000 000 pixels: with 1 MPix chunks the cuts fall between groups (test_mix_cuts).  Each entry is
# (class, h, w).  At level 1 the thin RGBA images the reference rejects there become opaque ones of the same size.
GROUPS = (
    ("split", (("translucent_rgba", 400, 300), ("rgb", 300, 500), ("gray_as_rgb", 200, 300), ("single_rgba", 50, 60),
               ("noise", 100, 70), ("rgb", 660, 1000))),
    ("rgb", (("gray_as_rgb", 400, 500), ("single_rgb", 50, 100), ("noise", 200, 300), ("rgb", 300, 400), ("rgb", 615, 1000))),
    ("opaque_dirty", (("opaque_rgba", 260, 300), ("dirty_clear_rgba", 40, 50), ("dirty_rgba", 300, 260), ("dirty_rgba", 500, 556),
                      ("opaque_rgba", 564, 1000))),
    ("stored_thin", (("stored_rgb_1x1", 1, 1), ("stored_rgba_1x1", 1, 1), ("thin_rgb_1xN", 1, 1399), ("thin_rgb_Nx1", 1823, 1),
                     ("thin_opaque_rgba", 50, 2), ("thin_single_rgba", 50, 2), ("thin_clear_rgba", 50, 3), ("wide_tile", 37, 1500),
                     ("thin_rgb_Nx1", 53814, 1), ("gray_as_rgb", 666, 666), ("largest_tile", 666, 666))),
    ("rgba", (("translucent_rgba", 500, 400), ("translucent_rgba", 300, 600), ("translucent_ramp", 4, 250),
              ("translucent_rgba", 619, 1000))),
    ("split2", (("single_rgb", 100, 100), ("translucent_rgba", 250, 400), ("gray_as_rgb", 300, 300), ("rgb", 400, 500),
                ("translucent_rgba", 600, 1000))),
)
GROUP_PX = 1_000_000


def make(cls, h, w, seed):
    return np.ascontiguousarray(GENS[CLASSES[cls][0]](h, w, seed))


def level_class(cls, level):
    """The class an entry of mix() has at `level`: the rejected thin RGBA images become opaque ones there."""
    return "thin_opaque_rgba" if CLASSES[cls][2][level] is None else cls


@lru_cache(maxsize=None)
def mix(level):
    """The batch at `level`: ([class], [pixels], group boundaries)."""
    classes, imgs, bounds = [], [], [0]
    for g, (_, items) in enumerate(GROUPS):
        for k, (cls, h, w) in enumerate(items):
            cls = level_class(cls, level)
            classes.append(cls)
            imgs.append(make(cls, h, w, 100 * g + k))
        bounds.append(len(imgs))
    return classes, imgs, bounds


def header(f):
    """(A, mode, single colour) of an .xpng file."""
    h0, h1 = struct.unpack_from("<II", f, 0)
    return (h1 >> 24) & 1, h0 >> 24, int(bool((h1 >> 24) & 2))


@lru_cache(maxsize=None)
def oracle_files(level):
    return tuple(po.encode(level, px) for px in mix(level)[1])


@lru_cache(maxsize=None)
def normalized(level):
    return tuple(po.normalize(px) for px in mix(level)[1])


def npx(px):
    return px.shape[0] * px.shape[1]


def split_groups(imgs, level):
    """Whether encode_issue splits a chunk of imgs into a level-1 and a level-2 group: at level 2, a chunk with an RGBA
    image that holds both a translucent image and an RGB (or opaque) image, each more than 4 bytes and not one colour."""
    if level != 2 or not any(px.shape[2] == 4 for px in imgs):
        return False
    fam = set()
    for px in imgs:
        n = po.normalize(px)
        flat = n.reshape(-1, n.shape[2])
        if n.size > 4 and not (flat == flat[0]).all():
            fam.add(n.shape[2])
    return fam == {3, 4}


def encode_chunks(imgs, level, lanes):
    """(chunks, k_image_offsets launches) of an encode call: one launch per chunk, two for a split chunk; none when level 7
    without RGBA takes the stored fast path."""
    if level == 7 and not any(px.shape[2] == 4 for px in imgs):
        return 0, 0
    cuts = restated_cuts([npx(px) for px in imgs], lanes)
    return len(cuts) - 1, sum(1 + split_groups(imgs[a:b], level) for a, b in zip(cuts, cuts[1:]))


def coded(f):
    """A file with tiles to decode (mode 1 or 2, not one colour)."""
    _, mode, single = header(f)
    return mode in (1, 2) and not single


def decode_chunks(files, dims, lanes):
    """(chunks, k_dec_tile_offsets launches) of a decode call whose entries decode dims[i] = (w, h) pixels each: one
    launch per chunk that holds a coded file."""
    cuts = restated_cuts([w * h for w, h in dims], lanes)
    return len(cuts) - 1, sum(any(coded(f) for f in files[a:b]) for a, b in zip(cuts, cuts[1:]))


CORPUS_PICK = (("2021.png", 1), ("juicy.png", 2), ("pigz-logo.png", 1), ("evil.png", 2), ("rodina.png", 2), ("pe4en_k.png", 1),
               ("weight_of_a_demultiplicator.png", 1), ("olaf.png", 2))


@lru_cache(maxsize=None)
def corpus():
    """Committed corpus images (RGB and RGBA), each coded at level 1 or 2: (files, normalised pixels)."""
    pxs = [load_png(os.path.join(CORPUS, name)) for name, _ in CORPUS_PICK]
    return tuple(po.encode(lv, px) for px, (_, lv) in zip(pxs, CORPUS_PICK)), tuple(po.normalize(px) for px in pxs)


# ------------------------------------------------------------------------------------------------------- CPU tests

def test_class_headers():
    """What each image class exercises: the oracle's header (A, mode, one colour) at every level, or a rejection."""
    for name, (gen, (h, w), want) in CLASSES.items():
        px = make(name, h, w, 3)
        for lv in (1, 2, 7):
            if want[lv] is None:
                with pytest.raises(ValueError):
                    po.encode(lv, px)
            else:
                assert header(po.encode(lv, px)) == want[lv], (name, lv)


@pytest.mark.parametrize("level", (1, 2, 7))
def test_mix_members_keep_their_class(level):
    """Every image of mix() has its class's header: the batch holds what GROUPS says it holds."""
    classes, _, _ = mix(level)
    for cls, f in zip(classes, oracle_files(level)):
        assert header(f) == CLASSES[cls][2][level], (cls, level)


@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("lanes", (2, 3))
def test_mix_cuts(level, lanes):
    """Six chunks, one per group, on two or three lanes: every lane runs at least two chunks of different kinds; at level 2
    the two mixed groups are split."""
    classes, imgs, bounds = mix(level)
    assert [sum(npx(px) for px in imgs[a:b]) for a, b in zip(bounds, bounds[1:])] == [GROUP_PX] * len(GROUPS)
    assert restated_cuts([npx(px) for px in imgs], lanes) == bounds
    chunks, launches = encode_chunks(imgs, level, lanes)
    assert chunks == len(GROUPS) > lanes
    kinds = [g for g, _ in GROUPS]
    for lane in range(lanes):
        seq = kinds[lane::lanes]
        assert len(seq) >= 2 and all(a != b for a, b in zip(seq, seq[1:]))
    split = [split_groups(imgs[a:b], level) for a, b in zip(bounds, bounds[1:])]
    assert split == ([True, False, True, False, False, True] if level == 2 else [False] * 6)
    assert launches == chunks + sum(split)


def test_restated_cuts_defaults():
    """With the default knobs (8 lanes, chunks of at least 32 MPix) a batch below 32 MPix is one chunk; above it, chunks
    of equal share that never split an image."""
    assert restated_cuts([1920 * 1080] * 15, 8, 32 * MPIX, 1 << 30) == [0, 15]
    assert restated_cuts([1920 * 1080] * 64, 8, 32 * MPIX, 1 << 30) == [0, 16, 32, 48, 64]
    assert restated_cuts([5, 1, 1, 1], 8, 1, 1 << 30) == [0, 1, 2, 4]        # the first image takes two shares of four
    assert restated_cuts([3 * MPIX, 1, 1], 2, MPIX, MPIX) == [0, 1, 3]      # an image above the chunk bound stays whole


def decode_order():
    """Files of mix() in an order that cuts into six chunks where lane 0 of two decodes a level-1 RGBA chunk, then a level-2
    RGB chunk, then a stored chunk: (files, normalised pixels)."""
    files, norms = [], []
    for level, g in ((1, 4), (1, 0), (2, 1), (2, 2), (7, 1), (2, 3)):
        a, b = mix(level)[2][g: g + 2]
        files += oracle_files(level)[a:b]
        norms += normalized(level)[a:b]
    return files, norms


def test_decode_order_cuts():
    files, norms = decode_order()
    cuts = restated_cuts([npx(n) for n in norms], 2)
    assert len(cuts) == 7
    lane0 = [[header(f) for f in files[a:b]] for a, b in zip(cuts[0::2], cuts[1::2])]
    assert all(h[:2] == (1, 1) for h in lane0[0])                                   # level-1 RGBA
    assert all(h[0] == 0 for h in lane0[1]) and any(h[1] == 2 for h in lane0[1])   # level-2 RGB
    assert all(h[1] == 7 for h in lane0[2])                                         # stored
    assert decode_chunks(files, [(n.shape[1], n.shape[0]) for n in norms], 2) == (6, 5)


def error_batch(level):
    """mix() at `level` with a thin translucent RGBA image in the third chunk (its opaque neighbour is 100 pixels smaller, so
    the cuts stay): (images, caller index of the thin image)."""
    classes, imgs, bounds = mix(level)
    g = bounds[2]
    assert classes[g] == "opaque_rgba" and npx(imgs[g]) == 78000
    bad = make("thin_translucent_rgba", 50, 2, 9)
    return list(imgs[:g]) + [make("opaque_rgba", 100, 779, 8), bad] + list(imgs[g + 1:]), g + 1


@pytest.mark.parametrize("level", (1, 2))
def test_error_batch_cuts(level):
    imgs, k = error_batch(level)
    cuts = restated_cuts([npx(px) for px in imgs], 2)
    assert len(cuts) == 7 and cuts[2] < k < cuts[3]
    with pytest.raises(ValueError):
        po.encode(level, imgs[k])


# ------------------------------------------------------------------------------------------------------- GPU helpers

def _codec(monkeypatch, lanes, family="lat"):
    """A codec whose calls cut 1 MPix chunks onto `lanes` lanes; family "pair" forces the batch decoder family."""
    for key, v in KNOBS.items():
        monkeypatch.setenv(key, v)
    monkeypatch.setenv("XPNGB_PIPE_LANES", str(lanes))
    if family == "pair":
        monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    else:
        monkeypatch.delenv("XPNGB_LAT_MAX_BLOCKS", raising=False)
    return xpng_b200.Codec(0)


def _run(cd, call, kernel=None, want=None, what=None):
    """call(); with a kernel named, under the profile, asserting that the call launched it `want` times."""
    if kernel is None:
        return call()
    cd.profile(True)
    try:
        r = call()
        got = cd.profile_report().get(kernel, (0.0, 0))[1]
    finally:
        cd.profile(False)
    assert got == want, (what, kernel, got, want)
    return r


def _order(name, cuts):
    """Host layouts of a batch: ascending, reversed, or interleaved (round robin over the chunks, so that every chunk's
    images sit between other chunks' images)."""
    n = cuts[-1]
    if name == "ascending":
        return list(range(n))
    if name == "reversed":
        return list(range(n))[::-1]
    spans = [range(a, b) for a, b in zip(cuts, cuts[1:])]
    return [s[r] for r in range(max(len(s) for s in spans)) for s in spans if r < len(s)]


def _layout(imgs, order):
    """Images packed at 16-byte offsets in the order `order`: (descriptors, bytes, buffer)."""
    n = len(imgs)
    descs = (_Image * n)()
    off = 0
    for i in order:
        h, w, c = imgs[i].shape
        descs[i].w, descs[i].h, descs[i].offset, descs[i].A, descs[i].mode = w, h, off, int(c == 4), 0
        off = (off + imgs[i].size + 15) & ~15
    buf = np.zeros(off + 16, np.uint8)
    for i in range(n):
        buf[descs[i].offset: descs[i].offset + imgs[i].size] = imgs[i].reshape(-1)
    return descs, off, buf


def _encode(cd, level, imgs, order, pix_dev, out_dev, hout=None):
    """encode_raw of imgs laid out in `order` into a device buffer of xpngb_encode_bound bytes, or into the host buffer
    hout (its last GUARD bytes excluded; a fresh one of the bound when None): (descriptors after the call, offsets,
    sizes, output bytes, capacity)."""
    import torch
    n = len(imgs)
    descs, total, buf = _layout(imgs, order)
    bound = int(xpng_b200.lib().xpngb_encode_bound(descs, n))
    if not out_dev and hout is None:
        hout = np.full(bound + GUARD, 0xA5, np.uint8)
    cap = bound if out_dev else len(hout) - GUARD
    dpix = torch.from_numpy(buf).cuda() if pix_dev else None
    dout = torch.empty(cap, dtype=torch.uint8, device="cuda") if out_dev else None
    torch.cuda.synchronize()
    offs, sizes = cd.encode_raw(level, descs, n, dpix.data_ptr() if pix_dev else buf.ctypes.data, total, pix_dev,
                                dout.data_ptr() if out_dev else hout.ctypes.data, cap, out_dev)
    return descs, list(offs), list(sizes), dout.cpu().numpy() if out_dev else hout, cap


def _check_encoded(want, descs, offs, sizes, out, cap, what):
    for i, f in enumerate(want):
        assert offs[i] % 16 == 0 and offs[i] + sizes[i] <= cap, (what, i)
        assert out[offs[i]: offs[i] + sizes[i]].tobytes() == f, (what, i)
        assert (descs[i].A, descs[i].mode) == header(f)[:2], (what, i)
    spans = sorted(zip(offs, sizes))
    assert all(a + s <= b for (a, s), (b, _) in zip(spans, spans[1:])), what
    if len(out) > cap:                     # host output: nothing written past the capacity
        assert (out[cap:] == 0xA5).all(), what


def _pack_files(files, out_bytes, out_order):
    """Files packed at 16-byte offsets; entry i's output at 16-byte offsets in the order out_order."""
    n = len(files)
    descs = (_Image * n)()
    foffs, fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
    fb = bytearray()
    for i, f in enumerate(files):
        foffs[i], fsizes[i] = len(fb), len(f)
        fb += f + b"\0" * (-len(f) % 16)
    poff = 0
    for i in out_order:
        descs[i].offset = poff
        poff += (out_bytes[i] + 15) & ~15
    return descs, foffs, fsizes, np.frombuffer(bytes(fb) + b"\0" * 16, np.uint8).copy(), len(fb), poff


def _decode(cd, files, out_bytes, out_order, files_dev, px_dev, boxes=None, szs=None):
    """decode_raw, decode_region_raw (boxes) or decode_resized_raw (szs) of files: (descriptors, output bytes)."""
    import torch
    n = len(files)
    descs, foffs, fsizes, fb, fsize, poff = _pack_files(files, out_bytes, out_order)
    dfiles = torch.from_numpy(fb).cuda() if files_dev else None
    dpx = torch.empty(poff + 16, dtype=torch.uint8, device="cuda") if px_dev else None
    hpx = None if px_dev else np.full(poff + GUARD, 0xA5, np.uint8)
    torch.cuda.synchronize()
    fptr = dfiles.data_ptr() if files_dev else fb.ctypes.data
    pptr = dpx.data_ptr() if px_dev else hpx.ctypes.data
    if szs is not None:
        cd.decode_resized_raw(descs, None, None, size_arr(szs), n, fptr, fsize, files_dev, foffs, fsizes, pptr, poff, px_dev)
    elif boxes is not None:
        cd.decode_region_raw(descs, rects(boxes), n, fptr, fsize, files_dev, foffs, fsizes, pptr, poff, px_dev)
    else:
        cd.decode_raw(descs, n, fptr, fsize, files_dev, foffs, fsizes, pptr, poff, px_dev)
    if px_dev:
        return descs, dpx.cpu().numpy()
    assert (hpx[poff:] == 0xA5).all()
    return descs, hpx


def _check_decode(cd, files, dims, wants, lanes, files_dev, px_dev, what, out_order=None, boxes=None, szs=None, count=True):
    """Decode files (whole, rectangles `boxes` or resized to `szs`) and compare entry i with wants[i].  dims[i] = (w, h):
    the pixels entry i decodes, by which the call cuts its chunks.  count: assert from the profile that every chunk
    holding a coded file ran."""
    chunks, want = decode_chunks(files, dims, lanes)
    assert chunks > lanes, (what, chunks)
    order = range(len(files)) if out_order is None else out_order
    descs, out = _run(cd, lambda: _decode(cd, files, [w.size for w in wants], order, files_dev, px_dev, boxes, szs),
                      "k_dec_tile_offsets" if count else None, want, what)
    for i, w in enumerate(wants):
        got = out[descs[i].offset: descs[i].offset + w.size].reshape(w.shape)
        assert np.array_equal(got, w), (what, i, None if boxes is None else boxes[i], None if szs is None else szs[i])


def _whole_dims(norms):
    return [(n.shape[1], n.shape[0]) for n in norms]     # a whole image, also resized, decodes all of it


def _random_boxes(rng, norms):
    boxes = []
    for n in norms:
        h, w = n.shape[:2]
        x, y = int(rng.integers(w)), int(rng.integers(h))
        boxes.append((x, y, int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1))))
    return boxes


def _region_dims(files, norms, boxes):
    """A region decode decodes the tiles its rectangle touches, a stored file only the rectangle."""
    dims = []
    for f, n, b in zip(files, norms, boxes):
        cover = b if header(f)[1] == 7 else region_tiles(n.shape[1], n.shape[0], b)[1]
        dims.append((cover[2], cover[3]))
    return dims


def _crops(norms, boxes):
    return [n[y: y + h, x: x + w] for n, (x, y, w, h) in zip(norms, boxes)]


def _random_sizes(rng, norms):
    """Output sizes from a quarter to twice each side, at most 600 (keeps the numpy reference quick)."""
    return [tuple(min(int(rng.integers(max(1, d // 4), 2 * d + 1)), 600) for d in (n.shape[1], n.shape[0])) for n in norms]


def _resized(norms, szs):
    return [resize_bilinear(n, w, h) for n, (w, h) in zip(norms, szs)]


def _all_files():
    """Every file of mix() at every level and the corpus files: (files, normalised pixels)."""
    cf, cn = corpus()
    return ([f for lv in (1, 2, 7) for f in oracle_files(lv)] + list(cf),
            [n for lv in (1, 2, 7) for n in normalized(lv)] + list(cn))


# ------------------------------------------------------------------------------------------------------- encode (GPU)

PLACEMENTS = {"host_host": (0, 0), "device_device": (1, 1), "host_device": (0, 1), "device_host": (1, 0)}


@gpu
@pytest.mark.parametrize("lanes", (2, 3))
@pytest.mark.parametrize("level", (1, 2, 7))
def test_encode_across_chunks(monkeypatch, level, lanes):
    """mix() in six chunks, in every buffer placement and, for host pixels, three layouts: each file equals the oracle's,
    each descriptor carries the file's A and mode, and the files are aligned, disjoint and inside the output."""
    _, imgs, bounds = mix(level)
    want = oracle_files(level)
    chunks, launches = encode_chunks(imgs, level, lanes)
    assert chunks == 6 > lanes
    cd = _codec(monkeypatch, lanes)
    try:
        for place, (pix_dev, out_dev) in PLACEMENTS.items():
            for k, layout in enumerate(("ascending", "reversed", "interleaved") if not pix_dev else ("interleaved",)):
                what = (level, lanes, place, layout)
                order = _order(layout, bounds)
                r = _run(cd, lambda: _encode(cd, level, imgs, order, pix_dev, out_dev),
                         "k_image_offsets" if place == "host_host" and k == 0 else None, launches, what)
                _check_encoded(want, *r, what)
    finally:
        cd.close()


@lru_cache(maxsize=None)
def _oriented_files(level, op):
    return tuple(po.encode(level, po.orient(op, px)) for px in mix(level)[1])


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_encode_oriented_across_chunks(monkeypatch, level):
    """encode_oriented of mix() with every op: each file equals the oracle's file of the turned or mirrored image."""
    _, imgs, _ = mix(level)
    _, launches = encode_chunks(imgs, level, 2)     # turned images keep their pixels, so the cuts stay
    cd = _codec(monkeypatch, 2)
    try:
        for k, op in enumerate(ALL_OPS):
            files = _run(cd, lambda: cd.encode_oriented(level, op, imgs), "k_image_offsets" if k == 0 else None, launches,
                         (level, op))
            want = _oriented_files(level, op)
            assert len(files) == len(want)
            for i, (g, w) in enumerate(zip(files, want)):
                assert g == w, (level, op, i)
    finally:
        cd.close()


# ------------------------------------------------------------------------------------------------------- decode (GPU)

@gpu
@pytest.mark.parametrize("family", ("lat", "pair"))
def test_decode_across_chunks(monkeypatch, family):
    """Both decoder families on two lanes.  decode_order: lane 0 decodes a level-1 RGBA chunk, a level-2 RGB chunk, then a
    stored chunk.  Then every file of mix() and the corpus in a random order, outputs in another: whole images, random
    rectangles and random sizes, with host and device buffers."""
    cd = _codec(monkeypatch, 2, family)
    rng = np.random.default_rng(20261021 + (family == "pair"))
    try:
        files, norms = decode_order()
        for files_dev, px_dev in ((0, 0), (1, 1)):
            _check_decode(cd, files, _whole_dims(norms), norms, 2, files_dev, px_dev, (family, "decode_order", files_dev),
                          count=not files_dev)
        af, an = _all_files()
        perm = rng.permutation(len(af))
        pf, pn = [af[k] for k in perm], [an[k] for k in perm]
        for files_dev, px_dev in ((0, 0), (1, 0)):
            _check_decode(cd, pf, _whole_dims(pn), pn, 2, files_dev, px_dev, (family, "all", files_dev, px_dev),
                          out_order=rng.permutation(len(pf)), count=not files_dev)
        boxes = _random_boxes(rng, pn)
        crops = _crops(pn, boxes)
        for files_dev, px_dev in ((0, 0), (0, 1)):
            _check_decode(cd, pf, _region_dims(pf, pn, boxes), crops, 2, files_dev, px_dev, (family, "region", files_dev, px_dev),
                          boxes=boxes, count=not px_dev)
        perm = rng.permutation(len(files))
        sf, sn = [files[k] for k in perm], [norms[k] for k in perm]
        szs = _random_sizes(rng, sn)
        resized = _resized(sn, szs)
        for files_dev, px_dev in ((0, 0), (1, 1)):
            _check_decode(cd, sf, _whole_dims(sn), resized, 2, files_dev, px_dev, (family, "resized", files_dev, px_dev),
                          szs=szs, count=not files_dev)
    finally:
        cd.close()


# ------------------------------------------------------------------------------------------------------- state (GPU)

def _steps():
    """Eight calls of different kinds and content for one codec, each checked against the oracle."""
    rng = np.random.default_rng(55)
    f1, n1 = list(oracle_files(1)), list(normalized(1))
    f2, n2 = list(oracle_files(2)), list(normalized(2))
    cf, cn = corpus()
    f7, n7 = list(oracle_files(7)) + list(cf), list(normalized(7)) + list(cn)
    boxes = _random_boxes(rng, n2)
    crops = _crops(n2, boxes)
    szs = _random_sizes(rng, n7)
    resized = _resized(n7, szs)

    def enc(level, place, layout):
        _, imgs, bounds = mix(level)
        return lambda cd: _check_encoded(oracle_files(level), *_encode(cd, level, imgs, _order(layout, bounds), *PLACEMENTS[place]),
                                         (level, place, layout))

    def oriented(cd):
        assert cd.encode_oriented(2, "r90", mix(2)[1]) == list(_oriented_files(2, "r90"))

    return [
        ("encode level 2", enc(2, "host_host", "interleaved")),
        ("decode level 1", lambda cd: _check_decode(cd, f1, _whole_dims(n1), n1, 2, 0, 0, "decode level 1", count=False)),
        ("encode level 7", enc(7, "device_device", "ascending")),
        ("region level 2", lambda cd: _check_decode(cd, f2, _region_dims(f2, n2, boxes), crops, 2, 1, 0, "region level 2",
                                                    boxes=boxes, count=False)),
        ("encode level 1", enc(1, "host_device", "reversed")),
        ("resized level 7 and corpus", lambda cd: _check_decode(cd, f7, _whole_dims(n7), resized, 2, 0, 1, "resized", szs=szs,
                                                                count=False)),
        ("decode level 2", lambda cd: _check_decode(cd, f2, _whole_dims(n2), n2, 2, 1, 1, "decode level 2", count=False)),
        ("oriented level 2", oriented),
    ]


@gpu
def test_state_from_earlier_calls(monkeypatch):
    """The same eight calls on one pipelined codec, then in reverse order on a fresh one: whatever a lane's scratch holds
    from an earlier call of another kind, every result equals the oracle's."""
    steps = _steps()
    for run in (steps, steps[::-1]):
        cd = _codec(monkeypatch, 2)
        try:
            for name, step in run:
                step(cd)
        finally:
            cd.close()


# ------------------------------------------------------------------------------------------------------- errors (GPU)

@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_thin_rgba_error_names_the_caller_index(monkeypatch, level):
    """A thin translucent RGBA image in the third chunk is refused under the caller's index, not its index in the chunk;
    the codec then encodes the batch without it."""
    imgs, k = error_batch(level)
    cd = _codec(monkeypatch, 2)
    try:
        for place in ("host_host", "device_device"):
            with pytest.raises(RuntimeError, match=rf"image {k}: RGBA tiles thinner than 4 pixels"):
                _encode(cd, level, imgs, range(len(imgs)), *PLACEMENTS[place])
        _, good, bounds = mix(level)
        _check_encoded(oracle_files(level), *_encode(cd, level, good, _order("interleaved", bounds), 0, 0), (level, "after"))
    finally:
        cd.close()


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_host_output_too_small(monkeypatch, level):
    """Host output that holds the first chunks but not the fourth, or all but its last byte, is refused and nothing is
    written at or past its end; output of exactly the packed size (every file rounded up to 16 bytes) is enough."""
    _, imgs, bounds = mix(level)
    want = oracle_files(level)
    packed = [sum((len(f) + 15) & ~15 for f in want[a:b]) for a, b in zip(bounds, bounds[1:])]
    cd = _codec(monkeypatch, 2)
    try:
        for cap in (sum(packed[:4]) - 16, sum(packed) - 1):
            hout = np.full(cap + GUARD, 0xA5, np.uint8)
            with pytest.raises(RuntimeError, match="output buffer too small"):
                _encode(cd, level, imgs, range(len(imgs)), 0, 0, hout)
            assert (hout[cap:] == 0xA5).all(), cap
        hout = np.full(sum(packed) + GUARD, 0xA5, np.uint8)
        _check_encoded(want, *_encode(cd, level, imgs, range(len(imgs)), 0, 0, hout), (level, "exact"))
    finally:
        cd.close()


# ------------------------------------------------------------------------------------------------------- pool (GPU)

@gpu
def test_pool_over_devices(monkeypatch):
    """shard.Pool over every device with the same knobs: the files equal the oracle's and the one-device pool's."""
    import torch
    from xpng_b200 import shard
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs two GPUs")
    for key, v in KNOBS.items():
        monkeypatch.setenv(key, v)
    monkeypatch.setenv("XPNGB_PIPE_LANES", "2")
    _, imgs, _ = mix(2)
    got = []
    for devs in ([0], list(range(ndev))):
        pool = shard.Pool(devs)
        try:
            files, _, _ = pool.encode(2, imgs)
            assert files == list(oracle_files(2)), devs
            for b, n in zip(pool.decode(files), normalized(2)):
                assert np.array_equal(b, n), devs
            got.append(files)
        finally:
            pool.close()
    assert got[0] == got[1]
