"""Resized decode (xpngb_decode_resized / Codec.decode_resized): each image or crop resampled to a requested size, then
written as its op leaves it, byte-identical to Pillow's Image.resize(size, Image.BILINEAR) of the crop.

resize_bilinear() restates Pillow's 8-bit bilinear resampling (Resample.c) in numpy.  It lives here rather than in oracle/,
which restates the format's reference code; it is pinned to the installed Pillow by the CPU tests below.
Without a GPU: resize_bilinear against PIL on seeded cases, as RGB images and channel by channel as "L" images.
On the GPU: every output equals po.orient(op, resize_bilinear(po.decode(f)[crop], w, h))."""
import ctypes as C
import hashlib
import json
import math
import os

import numpy as np
import pytest
from PIL import Image

from conftest import ROOT, make_case, manifest
from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import _Image, op_codes, rects, sizes as size_arr
from test_region import GENS, grid_rects, halfflat

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
PREC = 22                                           # Pillow's PRECISION_BITS for 8-bit images


# ---------------------------------------------------------------------------------------------------- the oracle

def _coeffs(inn, out):
    """Pillow's precompute_coeffs (bilinear, support 1) + normalize_coeffs_8bpc for one axis: per output coordinate the
    first input coordinate and ksize integer weights (zero past the window).  Python floats round every operation as
    x86-64 Pillow builds do."""
    scale = inn / out
    fs = max(scale, 1.0)
    support, ss = fs, 1.0 / fs
    ksize = int(math.ceil(support)) * 2 + 1
    xmins = np.zeros(out, np.int64)
    k = np.zeros((out, ksize), np.int64)
    for o in range(out):
        center = (o + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), inn)
        ws, ww = [], 0.0
        for t in range(xmax - xmin):
            x = abs((t + xmin - center + 0.5) * ss)
            w = 1.0 - x if x < 1.0 else 0.0
            ws.append(w)
            ww += w
        for t, w in enumerate(ws):
            k[o, t] = int(0.5 + (w / ww if ww != 0.0 else w) * (1 << PREC))
        xmins[o] = xmin
    return xmins, k


def _pass(px, out, axis):
    """One resampling pass along axis (0: vertical, 1: horizontal) of an (h, w, c) uint8 array."""
    inn = px.shape[axis]
    if inn == out:
        return px
    xmins, k = _coeffs(inn, out)
    src = np.moveaxis(px.astype(np.int64), axis, 0)
    acc = np.full((out,) + src.shape[1:], 1 << (PREC - 1), np.int64)
    for t in range(k.shape[1]):
        idx = np.minimum(xmins + t, inn - 1)            # weights past the window are 0
        acc += src[idx] * k[:, t].reshape((out,) + (1,) * (src.ndim - 1))
    return np.moveaxis(np.clip(acc >> PREC, 0, 255).astype(np.uint8), 0, axis)


def resize_bilinear(px, w, h):
    """Pillow's Image.resize((w, h), Image.BILINEAR) of the (h0, w0, c) uint8 array px, every channel on its own (as
    resizing each channel as an "L" image): the horizontal pass first, rounded to bytes, then the vertical pass.  Pillow
    12 runs the vertical pass first for images more than 100 times taller than wide that shrink vertically."""
    h0, w0 = px.shape[:2]
    if h < h0 and h0 > 100 * w0:
        return _pass(_pass(px, h, 0), w, 1)
    return _pass(_pass(px, w, 1), h, 0)


def pil_resize(px, w, h):
    return np.asarray(Image.fromarray(px).resize((w, h), Image.BILINEAR))


def pil_resize_channels(px, w, h):
    return np.stack([np.asarray(Image.fromarray(np.ascontiguousarray(px[:, :, c])).resize((w, h), Image.BILINEAR))
                     for c in range(px.shape[2])], axis=2)


# ---------------------------------------------------------------------------------------------------- oracle against PIL (CPU)

def oracle_cases():
    rng = np.random.default_rng(20261020)
    cases = [((1080, 1920), (224, 224)), ((1080, 1920), (1, 1)), ((1080, 7), (224, 224)), ((1333, 2111), (224, 224)),
             ((17, 3000), (40, 9)), ((5, 1920), (224, 3)), ((1, 1), (1, 1)), ((1, 1), (7, 5)), ((300, 1), (1, 300)),
             ((700, 7), (224, 224)), ((701, 7), (224, 224)), ((707, 7), (224, 708)), ((1080, 10), (5, 224)), ((1080, 11), (224, 224))]
    while len(cases) < 330:
        kind = len(cases) % 7
        h0, w0 = int(rng.integers(1, 401)), int(rng.integers(1, 401))
        if kind == 0:
            out = (1, 1)
        elif kind == 1:
            w0 = 1
            out = (int(rng.integers(1, 301)), int(rng.integers(1, 301)))
        elif kind == 2:
            out = (w0, h0)                                                   # identity
        elif kind == 3:
            out = (min(w0 + int(rng.integers(1, 300)), 300 + w0), min(h0 + int(rng.integers(1, 300)), 300 + h0))   # upscale
        elif kind == 4:
            out = (max(1, w0 // int(rng.integers(2, 9))), h0 + int(rng.integers(1, 200)))       # down in x, up in y
        elif kind == 5:                                                       # about 100 times taller than wide
            w0 = int(rng.integers(1, 4))
            h0 = int(rng.integers(95 * w0, 106 * w0 + 1))
            out = (int(rng.integers(1, 2 * w0 + 2)), int(rng.integers(1, 2 * h0)))
        else:
            out = (int(rng.integers(1, 301)), int(rng.integers(1, 301)))
        cases.append(((h0, w0), out))
    return cases


ORACLE_CASES = oracle_cases()


def test_oracle_case_count():
    assert len(ORACLE_CASES) >= 300
    tall = [(s, o) for s, o in ORACLE_CASES if o[1] < s[0] and s[0] > 100 * s[1] and o[0] != s[1]]
    assert len(tall) >= 20                              # the vertical-first order is exercised


@pytest.mark.parametrize("k", range(len(ORACLE_CASES)))
def test_resize_oracle_matches_pil(k):
    (h0, w0), (w, h) = ORACLE_CASES[k]
    rng = np.random.default_rng(k)
    px = rng.integers(0, 256, (h0, w0, 3), dtype=np.uint8)
    if k % 3 == 0:                                     # smooth content as well as noise
        px = np.cumsum(px.astype(np.int64), axis=1).astype(np.uint8)
    got = resize_bilinear(px, w, h)
    assert got.shape == (h, w, 3)
    assert np.array_equal(got, pil_resize(px, w, h))
    four = np.concatenate([px, rng.integers(0, 256, (h0, w0, 1), dtype=np.uint8)], axis=2)
    assert np.array_equal(resize_bilinear(four, w, h), pil_resize_channels(four, w, h))


# ---------------------------------------------------------------------------------------------------- resized decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def want_of(full, size, op, rect=None):
    if rect is not None:
        x, y, w, h = rect
        full = full[y: y + h, x: x + w]
    return po.orient(op or "tl", resize_bilinear(full, *size))


def check(codec, files, szs, boxes, ops, pil_every=0):
    """decode_resized of every entry against the oracle; every pil_every-th RGB entry also against PIL itself."""
    got = codec.decode_resized(files, szs, boxes, ops)
    fulls = {}
    for i, (f, z, g) in enumerate(zip(files, szs, got)):
        if f not in fulls:
            fulls[f] = po.decode(f)
        r = None if boxes is None else boxes[i]
        op = None if ops is None else ops[i]
        want = want_of(fulls[f], z, op, r)
        assert g.shape == want.shape and np.array_equal(g, want), (i, z, r, op)
        if pil_every and i % pil_every == 0 and g.shape[2] == 3:
            crop = fulls[f] if r is None else fulls[f][r[1]: r[1] + r[3], r[0]: r[0] + r[2]]
            assert np.array_equal(g, po.orient(op or "tl", pil_resize(crop, *z))), (i, z, r, op)
    return got


def size_kinds(w, h):
    """224 x 224, x1.7, mixed aspect (down in x, up in y), 1 x 1, 1 x h, identity."""
    return [(224, 224), (max(1, int(w * 1.7)), max(1, int(h * 1.7))), (max(1, w // 3), h * 2), (1, 1), (1, h), (w, h)]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("gen", sorted(GENS))
def test_resized_against_oracle(codec, gen, level):
    rng = np.random.default_rng(sorted(GENS).index(gen) * 3 + level + 200)
    h, w = 700, 1000                         # 2 x 2 tiles, as test_region_against_oracle
    f = po.encode(level, GENS[gen](h, w, 45))
    boxes = grid_rects(w, h, rng)
    entries = [(r, z) for r in boxes for z in size_kinds(r[2], r[3])]
    ops = [ALL_OPS[k % len(ALL_OPS)] for k in range(len(entries))]
    check(codec, [f] * len(entries), [z for _, z in entries], [r for r, _ in entries], ops, pil_every=5)
    check(codec, [f] * 6, size_kinds(w, h), None, None)                  # whole images, no op
    for k, op in enumerate(ALL_OPS):                                     # one entry per call
        r, z = entries[(7 * k + 3) % len(entries)]
        check(codec, [f], [z], [r], [op])


@gpu
@pytest.mark.parametrize("name", ("rgba_8192_s2", "rgb_4k_s1"))
def test_resized_large_golden(codec, name):
    entry = manifest()["synthetic"][name]
    px = make_case("synthetic", name, entry)
    h, w = px.shape[:2]
    boxes = [(0, 0, w, h), (0, 0, w, h), (1000, 1000, 1024, 1024), (w - 1000, 17, 1000, 777)]
    szs = [(224, 224), (1, 1), (224, 224), (300, 1200)]
    ops = ["tl", "mh", "r90", "mvh"]
    for lv in (1, 2):
        f = codec.encode(lv, [px])[0]
        assert hashlib.sha256(f).hexdigest() == entry["levels"][str(lv)]["sha256"]
        check(codec, [f] * len(boxes), szs, boxes, ops, pil_every=1)
        check(codec, [f], [(224, 224)], None, None)


@gpu
def test_identity_sizes_are_the_region_and_oriented_decode(codec):
    imgs = [synth.rgb(700, 1000, 31), synth.rgba(500, 460, 32), synth.rgb(1, 999, 33)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)] + [po.encode(2, imgs[0])]
    rng = np.random.default_rng(4)
    boxes = [grid_rects(im.shape[1], im.shape[0], rng)[-2] for im in imgs] + [(10, 20, 600, 400)]
    szs = [(r[2], r[3]) for r in boxes]
    plain = codec.decode_region(files, boxes)
    for a, b in zip(codec.decode_resized(files, szs, boxes), plain):
        assert a.shape == b.shape and a.tobytes() == b.tobytes()
    ops = ["r90", "mh", "r270", "tl"]
    for a, b in zip(codec.decode_resized(files, szs, boxes, ops), codec.decode_region(files, boxes, ops)):
        assert a.shape == b.shape and a.tobytes() == b.tobytes()
    whole = [(im.shape[1], im.shape[0]) for im in imgs] + [(1000, 700)]
    for a, b in zip(codec.decode_resized(files, whole, None, ops), codec.decode(files, ops)):
        assert a.shape == b.shape and a.tobytes() == b.tobytes()
    # identity entries next to resized ones in the same call stay byte-identical
    mixed = [szs[0], (224, 224), szs[2], (31, 7)]
    got = codec.decode_resized(files, mixed, boxes, ops)
    turned = codec.decode_region(files, boxes, ops)
    assert got[0].tobytes() == turned[0].tobytes() and got[2].tobytes() == turned[2].tobytes()
    assert np.array_equal(got[1], want_of(po.decode(files[1]), (224, 224), "mh", boxes[1]))


@gpu
def test_resized_mixed_batch(codec):
    imgs = [synth.rgb(900, 1300, 1), synth.rgba(500, 460, 2), synth.gray_as_rgb(300, 520, 3), synth.noise(90, 70, 4),
            np.full((700, 800, 3), 9, np.uint8), synth.rgb(1, 1399, 6), synth.rgb(1823, 1, 5), synth.rgba(333, 129, 7)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7, 1, 2, 2, 1, 7), imgs)]
    rng = np.random.default_rng(12)
    batch, boxes, szs, ops = [], [], [], []
    for f, im in zip(files, imgs):
        h, w = im.shape[:2]
        for k in range(4):
            x0, y0 = int(rng.integers(w)), int(rng.integers(h))
            r = (0, 0, w, h) if k == 0 else (x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1)))
            batch.append(f); boxes.append(r)
            szs.append((int(rng.integers(1, 400)), int(rng.integers(1, 400))) if k < 3 else (r[2], r[3]))
            ops.append(ALL_OPS[int(rng.integers(len(ALL_OPS)))])
    # crops more than 100 times taller than wide, shrunk vertically: Pillow's vertical-first order
    for f, r, z in ((files[0], (5, 0, 8, 900), (224, 224)), (files[6], (0, 0, 1, 1823), (3, 500)), (files[2], (7, 0, 2, 300), (9, 5))):
        batch.append(f); boxes.append(r); szs.append(z); ops.append("r90")
    perm = rng.permutation(len(batch))
    check(codec, [batch[k] for k in perm], [szs[k] for k in perm], [boxes[k] for k in perm], [ops[k] for k in perm], pil_every=3)


@gpu
def test_resized_batch_kernel_family(monkeypatch):
    """The pair decoders, three-tile walk and row-pitched un-predict (selected by batch size), forced on small inputs."""
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(8)
        for lv in (1, 2):
            for im in (synth.rgb(700, 1000, 81), synth.rgba(900, 700, 82), halfflat(700, 1000, 23)):
                h, w = im.shape[:2]
                f = po.encode(lv, im)
                boxes = grid_rects(w, h, rng)
                szs = [size_kinds(r[2], r[3])[k % 6] for k, r in enumerate(boxes)]
                ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in boxes]
                check(cd, [f] * len(boxes), szs, boxes, ops)
    finally:
        cd.close()


def rrc_boxes(rng, n, w=1920, h=1080):
    """RandomResizedCrop-style boxes: area share U(0.08, 1), aspect log-uniform in [3/4, 4/3], clipped to the frame."""
    out = []
    for _ in range(n):
        area = w * h * rng.uniform(0.08, 1.0)
        ar = math.exp(rng.uniform(math.log(3 / 4), math.log(4 / 3)))
        cw, ch = min(w, max(1, int(round(math.sqrt(area * ar))))), min(h, max(1, int(round(math.sqrt(area / ar)))))
        out.append((int(rng.integers(w - cw + 1)), int(rng.integers(h - ch + 1)), cw, ch))
    return out


@gpu
def test_resized_pipelined_chunks(monkeypatch):
    """64 sintel-like frames with one RandomResizedCrop-style box each, resized to 224 x 224 with a random op, cut into
    several chunks on three lanes (lanes are reused within the call), through the batch kernel family."""
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "config3_64.json")))
    frames = synth.sintel_batch(range(1000, 1064))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "3")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "3")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(66)
        boxes = rrc_boxes(rng, len(frames))
        ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in frames]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for k, f in enumerate(files):
                size, digest = gold[str(1000 + k)][str(lv)]
                assert len(f) == size and hashlib.sha256(f).hexdigest() == digest
            check(cd, files, [(224, 224)] * len(files), boxes, ops)
            check(cd, files[:16], [(224, 224)] * 16, None, None)
    finally:
        cd.close()


def pack(files, out_sizes, fill=0):
    """Files packed at 16-byte offsets, output offsets for out_sizes bytes each."""
    n = len(files)
    descs = (_Image * n)()
    foffs, fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
    fb, poff = bytearray(), 0
    for i, f in enumerate(files):
        foffs[i], fsizes[i] = len(fb), len(f)
        fb += f + b"\0" * (-len(f) % 16)
        descs[i].offset = poff
        poff += (out_sizes[i] + 15) & ~15
    return descs, foffs, fsizes, bytes(fb), poff


@gpu
def test_resized_device_resident_buffers(codec):
    import torch
    frames = [synth.rgb(720, 1280, 60), synth.rgba(600, 900, 61), synth.rgb(333, 517, 62), synth.rgba(64, 48, 63)]
    files = [po.encode(lv, f) for lv, f in zip((1, 1, 2, 7), frames)]
    szs = [(224, 224), (100, 333), (517, 1), (96, 80)]
    for boxes in ([(100, 37, 600, 500), (0, 444, 900, 156), (17, 3, 1, 300), (3, 5, 41, 29)], None):
        for ops in (["r90", "mh", "r270", "mv"], None):
            nbytes = [w * h * f.shape[2] for (w, h), f in zip(szs, frames)]
            descs, foffs, fsizes, fb, poff = pack(files, nbytes)
            dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
            dpx = torch.zeros(poff, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            codec.decode_resized_raw(descs, None if ops is None else op_codes(ops), None if boxes is None else rects(boxes),
                                     size_arr(szs), len(files), dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dpx.data_ptr(), poff, 1)
            out = dpx.cpu().numpy()
            for i, f in enumerate(files):
                want = want_of(po.decode(f), szs[i], None if ops is None else ops[i], None if boxes is None else boxes[i])
                got = out[descs[i].offset: descs[i].offset + want.size].reshape(want.shape)
                assert np.array_equal(got, want), (i, boxes, ops)


@gpu
def test_resized_failures(codec):
    px = synth.rgb(600, 700, 5)
    f = po.encode(1, px)

    def call(files, szs, boxes=None, ops=None, cap_delta=0, offset=None):
        """decode_resized_raw into a sentinel-filled host buffer; the buffer is returned with the exception, if any."""
        nb = [max(1, w) * max(1, h) * 3 if 0 < w <= 1 << 24 and 0 < h <= 1 << 24 else 16 for w, h in szs]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        if offset is not None:
            descs[len(files) - 1].offset = offset
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, 0xA5, np.uint8)
        err = None
        try:
            codec.decode_resized_raw(descs, None if ops is None else (C.c_int * len(ops))(*ops), None if boxes is None else rects(boxes),
                                     size_arr(szs), len(files), fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data,
                                     poff + cap_delta, 0)
        except RuntimeError as e:
            err = str(e)
        return err, out

    bad_sizes = [(0, 10), (10, 0), ((1 << 24) + 1, 1), (1, (1 << 24) + 1), (2 ** 32 - 1, 5)]
    for z in bad_sizes:
        err, out = call([f, f], [(10, 10), z])
        assert err is not None and "entry 1" in err and "output size" in err, (z, err)
        assert (out == 0xA5).all(), z
    err, out = call([f, f], [(10, 10), (224, 224)], ops=[0, 9])
    assert "entry 1: unknown orientation op" in err and (out == 0xA5).all()
    err, out = call([f, f], [(10, 10), (224, 224)], boxes=[(0, 0, 5, 5), (0, 0, 701, 10)])
    assert "entry 1" in err and (out == 0xA5).all()
    err, out = call([f], [(224, 224)], cap_delta=-1)                       # output past pixels_cap (not the crop size)
    assert "exceed" in err and (out == 0xA5).all()
    err, out = call([f, f], [(5, 5), (224, 224)], offset=8 + 80)           # misaligned output offset
    assert "file 1" in err and "multiple of 16" in err and (out == 0xA5).all()
    descs, foffs, fsizes, fb, poff = pack([f], [224 * 224 * 3])
    fa = np.frombuffer(fb, np.uint8)
    out = np.full(poff + 16, 0xA5, np.uint8)
    assert xpng_b200.lib().xpngb_decode_resized(codec._h, None, descs, None, None, 1, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                                out.ctypes.data, poff, 0) != 0
    assert "null argument" in codec._err() and (out == 0xA5).all()
    with pytest.raises(RuntimeError, match="entry 1"):
        codec.decode_resized([f, f], [(5, 5), (0, 3)])
    # and the context still decodes afterwards
    assert np.array_equal(codec.decode_resized([f], [(224, 224)], None, ["mh"])[0], want_of(px, (224, 224), "mh"))
