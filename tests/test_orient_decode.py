"""Oriented decode (xpngb_decode_oriented / Codec.decode(ops=) / Codec.decode_region(ops=)): each entry written as its op
(tool --<op>) leaves the whole image or the crop, one op per entry in one call.

Without a GPU: the inverse-op table against the oracle's restatement of the reference tool.
On the GPU: every output equals po.orient(op, po.decode(f)[crop]) of the pinned CPU oracle."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import ROOT, make_case, manifest
from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import OPS, _Image, op_codes, rects
from test_region import GENS, grid_rects, halfflat

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)


# ---------------------------------------------------------------------------------------------------- op table (CPU)

def test_inverse_op_undoes_every_op():
    px = np.random.default_rng(1).integers(0, 256, (37, 53, 4), dtype=np.uint8)
    assert sorted(ALL_OPS) == sorted(OPS)
    for op in ALL_OPS:
        assert np.array_equal(po.orient(xpng_b200.inverse_op(op), po.orient(op, px)), px), op
    assert [xpng_b200.inverse_op(op) for op in ALL_OPS] == ["r270", "r90", "mv", "mh", "mvh", "tl", "tr"]


def test_unknown_op_names_are_refused():
    with pytest.raises(ValueError):
        xpng_b200.inverse_op("flip")
    with pytest.raises(ValueError, match="'r180'"):
        op_codes(["r90", "r180"])
    assert list(op_codes(ALL_OPS)) == [OPS[o] for o in ALL_OPS]


# ---------------------------------------------------------------------------------------------------- oriented decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def want_of(full, op, rect=None):
    if rect is not None:
        x, y, w, h = rect
        full = full[y: y + h, x: x + w]
    return po.orient(op, full)


def check(codec, files, boxes, ops):
    """decode_region (boxes) or decode (boxes None) with ops, every entry against the oracle."""
    got = codec.decode(files, ops) if boxes is None else codec.decode_region(files, boxes, ops)
    fulls = {}
    for i, (f, op, g) in enumerate(zip(files, ops, got)):
        if f not in fulls:
            fulls[f] = po.decode(f)
        want = want_of(fulls[f], op, None if boxes is None else boxes[i])
        assert g.shape == want.shape and np.array_equal(g, want), (i, op, None if boxes is None else boxes[i])
    return got


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("gen", sorted(GENS))
def test_oriented_against_oracle(codec, gen, level):
    rng = np.random.default_rng(sorted(GENS).index(gen) * 3 + level + 100)
    h, w = 700, 1000                         # 2 x 2 tiles, as test_region_against_oracle
    f = po.encode(level, GENS[gen](h, w, 43))
    boxes = grid_rects(w, h, rng)
    # every op on every rectangle of one file in one call
    entries = [(r, op) for r in boxes for op in ALL_OPS]
    check(codec, [f] * len(entries), [r for r, _ in entries], [op for _, op in entries])
    check(codec, [f] * len(ALL_OPS), None, ALL_OPS)             # whole images
    for op in ALL_OPS:                                          # one entry per call
        check(codec, [f], None, [op])
        for r in boxes:
            check(codec, [f], [r], [op])


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_round_trip_of_encode_oriented(codec, level):
    imgs = [synth.rgb(600, 911, 21), synth.rgba(450, 300, 22), synth.gray_as_rgb(333, 500, 23), synth.rgba(7, 1301, 24)]
    for op in ALL_OPS:
        files = codec.encode_oriented(level, op, imgs)
        back = codec.decode(files, [xpng_b200.inverse_op(op)] * len(files))
        for b, im in zip(back, imgs):
            assert b.shape == po.normalize(im).shape and np.array_equal(b, po.normalize(im)), (op, level, im.shape)


@gpu
def test_mixed_batch_one_call(codec):
    imgs = [synth.rgb(900, 1300, 1), synth.rgba(500, 460, 2), synth.gray_as_rgb(300, 520, 3), synth.noise(90, 70, 4),
            np.full((700, 800, 3), 9, np.uint8), synth.rgb(1, 1399, 6), synth.rgb(1823, 1, 5), synth.rgba(333, 129, 7)]
    levels = (1, 2, 7, 1, 2, 2, 1, 7)
    files = [po.encode(lv, im) for lv, im in zip(levels, imgs)]
    rng = np.random.default_rng(11)
    batch, boxes, ops = [], [], []
    for f, im in zip(files, imgs):
        h, w = im.shape[:2]
        for k in range(4):
            if k == 0:
                r = (0, 0, w, h)
            else:
                x0, y0 = int(rng.integers(w)), int(rng.integers(h))
                r = (x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1)))
            batch.append(f); boxes.append(r); ops.append(ALL_OPS[int(rng.integers(len(ALL_OPS)))])
    perm = rng.permutation(len(batch))
    check(codec, [batch[k] for k in perm], [boxes[k] for k in perm], [ops[k] for k in perm])
    wops = [ALL_OPS[k % len(ALL_OPS)] for k in range(len(files))]
    check(codec, files, None, wops)
    check(codec, files[::-1], None, wops)


@gpu
def test_copy_ops_are_the_unoriented_decode(codec):
    imgs = [synth.rgb(700, 1000, 31), synth.rgba(500, 460, 32), synth.rgb(1, 999, 33)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)] + [po.encode(2, imgs[0])]
    rng = np.random.default_rng(4)
    for op in ("tl", "tr"):
        plain = codec.decode(files)
        for a, b in zip(codec.decode(files, [op] * len(files)), plain):
            assert a.shape == b.shape and a.tobytes() == b.tobytes()
        # the last tile column (whole tiles: decoded in place), and a rectangle that is not made of whole tiles
        boxes = [grid_rects(im.shape[1], im.shape[0], rng)[-2] for im in imgs] + [(10, 20, 600, 400)]
        plain = codec.decode_region(files, boxes)
        for a, b in zip(codec.decode_region(files, boxes, [op] * len(files)), plain):
            assert a.shape == b.shape and a.tobytes() == b.tobytes()
    # mixed with turned entries in the same call, the copy entries stay byte-identical
    ops = ["tl", "r90", "tr", "mvh"]
    got = codec.decode(files, ops)
    plain = codec.decode(files)
    assert got[0].tobytes() == plain[0].tobytes() and got[2].tobytes() == plain[2].tobytes()
    assert np.array_equal(got[1], po.orient("r90", plain[1])) and np.array_equal(got[3], po.orient("mvh", plain[3]))


@gpu
def test_oriented_batch_kernel_family(monkeypatch):
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
                ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in boxes]
                check(cd, [f] * len(boxes), boxes, ops)
                check(cd, [f] * len(ALL_OPS), None, ALL_OPS)
    finally:
        cd.close()


@gpu
def test_oriented_pipelined_chunks(monkeypatch):
    """64 sintel-like frames with one seeded 224 x 224 crop and a random op each, then whole frames with random ops, cut
    into several chunks on three lanes (lanes are reused within the call), through the batch kernel family."""
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "config3_64.json")))
    frames = synth.sintel_batch(range(1000, 1064))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "3")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "3")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(65)
        boxes = [(int(rng.integers(1920 - 224)), int(rng.integers(1080 - 224)), 224, 224) for _ in frames]
        ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in frames]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for k, f in enumerate(files):
                size, digest = gold[str(1000 + k)][str(lv)]
                assert len(f) == size and hashlib.sha256(f).hexdigest() == digest
            check(cd, files, boxes, ops)
            check(cd, files[:16], None, ops[16:32])
    finally:
        cd.close()


def pack(files, out_sizes):
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
def test_oriented_device_resident_buffers(codec):
    import torch
    frames = [synth.rgb(720, 1280, 60), synth.rgba(600, 900, 61), synth.rgb(333, 517, 62), synth.rgba(64, 48, 63)]
    files = [po.encode(lv, f) for lv, f in zip((1, 1, 2, 7), frames)]
    for boxes in ([(100, 37, 600, 500), (0, 444, 900, 156), (17, 3, 1, 300), (3, 5, 41, 29)], None):
        ops = ["r90", "mh", "r270", "r90"]
        sizes = [(f.shape[0] * f.shape[1] if boxes is None else boxes[i][2] * boxes[i][3]) * f.shape[2] for i, f in enumerate(frames)]
        descs, foffs, fsizes, fb, poff = pack(files, sizes)
        dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
        dpx = torch.zeros(poff, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        codec.decode_oriented_raw(descs, op_codes(ops), None if boxes is None else rects(boxes), len(files), dfiles.data_ptr(), len(fb), 1,
                                  foffs, fsizes, dpx.data_ptr(), poff, 1)
        out = dpx.cpu().numpy()
        for i, f in enumerate(files):
            want = want_of(po.decode(f), ops[i], None if boxes is None else boxes[i])
            assert (descs[i].w, descs[i].h) == (frames[i].shape[1], frames[i].shape[0])      # descriptors are not swapped
            got = out[descs[i].offset: descs[i].offset + want.size].reshape(want.shape)
            assert np.array_equal(got, want), (i, boxes)


@gpu
@pytest.mark.parametrize("name", ("rgba_8192_s2", "rgb_4k_s1"))
def test_oriented_large_golden(codec, name):
    entry = manifest()["synthetic"][name]
    px = make_case("synthetic", name, entry)
    h, w = px.shape[:2]
    boxes = [(0, 0, w, h), (w - 1000, 17, 1000, 777), (1000, 1000, 1024, 1024)]
    for lv in (1, 2):
        f = codec.encode(lv, [px])[0]
        assert hashlib.sha256(f).hexdigest() == entry["levels"][str(lv)]["sha256"]
        full = po.decode(f)
        for op in ("r90", "r270", "mvh"):
            got = codec.decode_region([f] * len(boxes), boxes, [op] * len(boxes))
            for r, g in zip(boxes, got):
                assert np.array_equal(g, want_of(full, op, r)), (name, lv, op, r)
        assert np.array_equal(codec.decode([f], ["r90"])[0], po.orient("r90", full))


@gpu
def test_stored_rgba_at_unaligned_offset(codec):
    """A level-7 RGBA file whose pixels start at an odd byte address: k_orient moves them byte by byte."""
    f7 = po.encode(7, synth.rgba(130, 201, 71))
    assert po.peek(f7)[2:] == (1, 7) and len(f7) == 8 + 130 * 201 * 4      # stored, alpha kept
    img = po.decode(f7)
    other = po.encode(1, synth.rgb(70, 90, 72))
    boxes = [(0, 0, 201, 130), (5, 9, 64, 65), (0, 0, 201, 130)]
    ops = ["r90", "mvh", "mv"]
    for lead in (1, 2, 3):
        head = bytes(lead) + f7
        head += bytes(-len(head) % 16)
        fb = head + other + bytes(16)
        n = 4
        foffs = (C.c_uint64 * n)(lead, lead, lead, len(head))
        fsizes = (C.c_uint64 * n)(len(f7), len(f7), len(f7), len(other))
        descs = (_Image * n)()
        sizes = [r[2] * r[3] * 4 for r in boxes] + [70 * 90 * 3]
        poff = 0
        for i, s in enumerate(sizes):
            descs[i].offset = poff
            poff += (s + 15) & ~15
        out = np.zeros(poff + 16, np.uint8)
        arr = np.frombuffer(fb, np.uint8)
        codec.decode_oriented_raw(descs, op_codes(ops + ["r270"]), rects(boxes + [(0, 0, 90, 70)]), n, arr.ctypes.data, len(fb), 0,
                                  foffs, fsizes, out.ctypes.data, poff, 0)
        for i, (r, op) in enumerate(zip(boxes, ops)):
            want = want_of(img, op, r)
            assert np.array_equal(out[descs[i].offset: descs[i].offset + want.size].reshape(want.shape), want), (lead, i)
        want = po.orient("r270", po.decode(other))
        assert np.array_equal(out[descs[3].offset: descs[3].offset + want.size].reshape(want.shape), want)


@gpu
def test_oriented_failures(codec):
    px = synth.rgb(600, 700, 5)
    f = po.encode(1, px)
    for bad_op in (7, -1, 1 << 20):
        args, keep = raw_args([f, f], [0, bad_op], None)
        with pytest.raises(RuntimeError, match="entry 1: unknown orientation op"):
            codec.decode_oriented_raw(*args)
    descs, ops, ra, n, fptr, fsize, fdev, foffs, fsizes, pptr, pcap, pdev = args
    assert xpng_b200.lib().xpngb_decode_oriented(codec._h, None, descs, ra, n, C.c_void_p(fptr), fsize, fdev, foffs, fsizes,
                                                 C.c_void_p(pptr), pcap, pdev) != 0
    assert "null argument" in codec._err()
    # misaligned output offset, output past pixels_cap (a quarter turn writes the same byte count)
    (descs, ops, ra, n, fptr, fsize, fdev, foffs, fsizes, pptr, pcap, pdev), keep = raw_args([f], [0], [(10, 10, 100, 50)])
    descs[0].offset = 8
    with pytest.raises(RuntimeError, match="multiple of 16"):
        codec.decode_oriented_raw(descs, ops, ra, n, fptr, fsize, fdev, foffs, fsizes, pptr, pcap, pdev)
    descs[0].offset = 0
    with pytest.raises(RuntimeError, match="exceed"):
        codec.decode_oriented_raw(descs, ops, ra, n, fptr, fsize, fdev, foffs, fsizes, pptr, 100 * 50 * 3 - 1, pdev)
    args, keep = raw_args([f], [1], None)
    args = list(args); args[10] -= 1
    with pytest.raises(RuntimeError, match="exceed"):
        codec.decode_oriented_raw(*args)
    with pytest.raises(RuntimeError, match="entry 1"):
        codec.decode_region([f, f], [(0, 0, 5, 5), (0, 0, 701, 10)], ["r90", "r90"])
    bad = bytearray(f); bad[9] ^= 0xFF; bad[10] ^= 0x7F            # first tile's size word
    for boxes in ([(500, 400, 50, 50)], None):
        with pytest.raises(RuntimeError):
            if boxes is None:
                codec.decode([bytes(bad)], ["r270"])
            else:
                codec.decode_region([bytes(bad)], boxes, ["r270"])
    # and the context still decodes afterwards
    assert np.array_equal(codec.decode([f], ["mh"])[0], po.orient("mh", px))


def raw_args(files, ops, boxes):
    """Host-buffer arguments of decode_oriented_raw, and the buffers they point into (the caller keeps them alive)."""
    sizes = []
    for i, f in enumerate(files):
        w, h, A = po.peek(f)[:3]
        sizes.append((w * h if boxes is None else boxes[i][2] * boxes[i][3]) * (3 + int(A)))
    descs, foffs, fsizes, fb, poff = pack(files, sizes)
    fa = np.frombuffer(fb, np.uint8)
    out = np.zeros(poff + 16, np.uint8)
    return (descs, (C.c_int * len(ops))(*ops), None if boxes is None else rects(boxes), len(files), fa.ctypes.data, len(fb), 0,
            foffs, fsizes, out.ctypes.data, poff, 0), (fa, out)
