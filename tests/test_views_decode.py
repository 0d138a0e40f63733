"""Multi-view decode: entries of one call that read the same file (equal offset and size) decode its tiles once, into one
shared window, and Codec.decode_views returns every view of a multi-crop batch from one call.

The reference for the shared path is the library's own per-entry path, which a call still takes when each entry's file
sits at its own offset: both calls must give the same bytes, and the shared call must decode fewer tiles."""
import ctypes as C
import random

import numpy as np
import pytest
from PIL import Image

from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import (_Image, augment_array, augment_params, blur_array, color_array, filter_codes, op_codes, rects, region_tiles,
                             sizes as size_arr, tensor_format)
from test_blur_decode import DinoGaussianBlur, DinoSolarization, _replay_view, random_blur
from test_color_decode import random_col
from test_resampled_decode import FILTERS
from test_tensor_decode import IMAGENET

gpu = pytest.mark.gpu
ALL_OPS = ("r90", "r270", "mv", "mh", "mvh", "tl", "tr")
ENTRY_POINTS = ("region", "oriented", "resized", "tensor", "resampled", "color", "blur", "augment")
AUG_PROGRAMS = ([("Rotate", 12.0)], [("ShearX", 0.2)], [("Posterize", 5.0)], [("Equalize", 0.0)], [("AutoContrast", 0.0)],
                [("Brightness", 0.4)], [("Sharpness", -0.3)], [("Solarize", 100.0)], [("Invert", 0.0)],
                [("Color", 0.5), ("Contrast", -0.2)])


def pack(files, out_sizes, share):
    """Files at 16-byte offsets and 16-byte aligned output offsets.  share: an object that appears in several entries is
    packed once and its entries share its offset (the library then decodes it once); otherwise every entry's file is packed
    at its own offset, the per-entry path."""
    n = len(files)
    descs = (_Image * n)()
    foffs, fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
    fb, poff, seen = bytearray(), 0, {}
    for i, f in enumerate(files):
        if share and id(f) in seen:
            foffs[i] = seen[id(f)]
        else:
            foffs[i] = seen[id(f)] = len(fb)
            fb += f + b"\0" * (-len(f) % 16)
        fsizes[i] = len(f)
        descs[i].offset = poff
        poff += (out_sizes[i] + 15) & ~15
    return descs, foffs, fsizes, bytes(fb), poff


def bare_codec():
    """A Codec without a device context: enough for the host-side argument checks and packing."""
    cd = xpng_b200.Codec.__new__(xpng_b200.Codec)
    cd._h = C.c_void_p()
    cd.device = 0
    return cd


# ---------------------------------------------------------------------------------------------------- host only

def test_pack_files_shares_repeated_objects():
    a, b = po.encode(1, synth.rgb(40, 50, 1)), po.encode(2, synth.rgba(30, 20, 2))
    b2 = bytes(bytearray(b))   # equal bytes, another object: packed again
    assert b2 == b and b2 is not b
    files = [a, b, a, b2, b, a]
    descs, foffs, fsizes, fb, off, _, _ = bare_codec()._pack_files(files)
    assert foffs[0] == foffs[2] == foffs[5] and foffs[1] == foffs[4]
    assert len({foffs[0], foffs[1], foffs[3]}) == 3
    assert off == ((len(a) + 15) & ~15) + 2 * ((len(b) + 15) & ~15)
    for i, f in enumerate(files):
        assert fsizes[i] == len(f) and bytes(fb[foffs[i]: foffs[i] + len(f)]) == f
        assert (descs[i].w, descs[i].h, descs[i].A) == ((50, 40, 0) if f is a else (20, 30, 1))


def test_decode_views_argument_errors():
    cd = bare_codec()
    files = [po.encode(1, synth.rgb(60, 80, 3)), po.encode(1, synth.rgb(70, 90, 4))]
    cases = [
        ([dict(sizes=[(8, 8)] * 2, bogus=1)], "view 0: unknown key 'bogus'"),
        ([dict(), dict(sizes=[(8, 8)] * 2, crop=None)], "view 1: unknown key 'crop'"),
        ([dict(boxes=[(0, 0, 9, 9)] * 2), dict(sizes=[(8, 8)])], "view 1: one size per file"),
        ([dict(boxes=[(0, 0, 9, 9)])], "view 0: one box per file"),
        ([dict(boxes=[(0, 0, 9, 9)] * 2, ops=["tl"] * 3)], "view 0: one op per file"),
        ([dict(boxes=[(0, 0, 9, 9)] * 2), dict(boxes=[(0, 0, 9, 9)] * 2, filters="bicubic")], "view 1: filters and windows need sizes"),
        ([dict(sizes=[(8, 8)] * 2, windows=[(0, 0, 4, 4)] * 2), dict(windows=[(0, 0, 4, 4)] * 2)], "view 1: filters and windows need sizes"),
        ([dict(sizes=[(8, 8)] * 2, filters=["bicubic"])], "view 0: one filter per file"),
        ([dict(sizes=[(8, 8)] * 2, filters="nearest")], "view 0: unknown resampling filter"),
        ([dict(sizes=[(8, 8), (8, 9)])], "view 0: entries have different output shapes"),
        ([dict(sizes=[(8, 8)] * 2), dict()], "view 1: entries have different output shapes"),   # whole 80x60 and 90x70
        ([dict(boxes=[(0, 0, 9, 5)] * 2, ops=["tl", "r90"])], "view 0: entries have different output shapes"),
    ]
    for views, msg in cases:
        with pytest.raises(ValueError, match=msg.replace("(", r"\(")):
            cd.decode_views(files, views)
    with pytest.raises(ValueError, match="at least one"):
        cd.decode_views(files, [])
    with pytest.raises(ValueError, match="file 1: not an .xpng header"):
        cd.decode_views([files[0], b"\0" * 4], [dict()])


# ---------------------------------------------------------------------------------------------------- on the GPU

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def interleaved(rng, n_a=30, n_b=8):
    """File indices a = 0, b = 1, c = 2 beginning a, b, a, c, b, a: a has n_a entries, b n_b, c one."""
    seq = [0, 1, 0, 2, 1, 0]
    rest = [0] * (n_a - 3) + [1] * (n_b - 2)
    rng.shuffle(rest)
    return seq + rest


def random_box(rng, w, h):
    x, y = int(rng.integers(0, w)), int(rng.integers(0, h))
    return (x, y, int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1)))


def entries(rng, idx, heads, alpha_kept):
    """Per-entry arguments of every entry point for entries reading files idx.  alpha_kept: the output keeps alpha, so
    RGBA entries get no grayscale, solarize or augment program (the library refuses them)."""
    n = len(idx)
    boxes = [random_box(rng, heads[k][0], heads[k][1]) for k in idx]
    ops = [ALL_OPS[j % 7] for j in range(n)]
    szs = [(int(rng.integers(1, 160)), int(rng.integers(1, 160))) for _ in range(n)]
    wins = [random_box(rng, *z) for z in szs]
    filters = [FILTERS[j % 5] for j in range(n)]
    plain = [alpha_kept and heads[k][2] for k in idx]   # RGBA entries whose output keeps alpha
    cols = [random_col(rng, gray_ok=not p) if j % 3 else None for j, p in enumerate(plain)]
    blurs = [random_blur(rng, not p) if j % 2 else None for j, p in enumerate(plain)]
    augs = []
    for j, p in enumerate(plain):
        w, h = wins[j][2:]
        if ops[j] in ("r90", "r270"):
            w, h = h, w
        augs.append(None if p or j % 4 == 0 else augment_params(AUG_PROGRAMS[j % len(AUG_PROGRAMS)], (w, h), "bilinear"))
    return dict(boxes=boxes, ops=ops, szs=szs, wins=wins, filters=filters, cols=cols, blurs=blurs, augs=augs)


def out_hw(ep, e, j, full_hw):
    if ep in ("resampled", "color", "blur", "augment"):
        w, h = e["wins"][j][2:]
    elif ep in ("resized", "tensor"):
        w, h = e["szs"][j]
    else:
        w, h = e["boxes"][j][2:]
    return (w, h) if e["ops"][j] in ("r90", "r270") else (h, w)


def run(cd, ep, files, e, nb, fmt, share, dev=False):
    """One call of entry point ep; returns every entry's output bytes, concatenated, and the call's last_tiles.  The
    padding between entries belongs to no entry: with host buffers a call may copy the device's padding bytes back or
    not, depending on how its chunks fall, so it is not compared."""
    import torch
    n = len(files)
    descs, foffs, fsizes, fb, poff = pack(files, nb, share)
    fa = np.frombuffer(fb, np.uint8)
    ra, oa, sa, wa = rects(e["boxes"]), op_codes(e["ops"]), size_arr(e["szs"]), rects(e["wins"])
    fl = filter_codes(e["filters"], n)
    ca, ba, aa = color_array(e["cols"], n), blur_array(e["blurs"], n), augment_array(e["augs"], n)
    if dev:
        dfiles = torch.from_numpy(fa.copy()).cuda()
        dout = torch.full((poff + 16,), 0xA5, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        src, out, on = (dfiles.data_ptr(), dout.data_ptr(), 1)
    else:
        hout = np.full(poff + 16, 0xA5, np.uint8)
        src, out, on = (fa.ctypes.data, hout.ctypes.data, 0)
    io = (n, src, len(fb), on, foffs, fsizes, out, poff, on)
    if ep == "region":
        cd.decode_region_raw(descs, ra, *io)
    elif ep == "oriented":
        cd.decode_oriented_raw(descs, oa, ra, *io)
    elif ep == "resized":
        cd.decode_resized_raw(descs, oa, ra, sa, *io)
    elif ep == "tensor":
        cd.decode_tensor_raw(fmt, descs, oa, ra, sa, *io)
    elif ep == "resampled":
        cd.decode_resampled_raw(fmt, descs, fl, oa, ra, sa, wa, *io)
    elif ep == "color":
        cd.decode_color_raw(fmt, descs, fl, oa, ra, sa, wa, ca, *io)
    elif ep == "blur":
        cd.decode_blur_raw(fmt, descs, fl, oa, ra, sa, wa, ca, ba, *io)
    else:
        cd.decode_augment_raw(fmt, descs, fl, oa, ra, sa, wa, ca, ba, aa, *io)
    buf = dout.cpu().numpy() if dev else hout
    return np.concatenate([buf[d.offset: d.offset + b] for d, b in zip(descs, nb)]), cd.last_tiles


def bbox(boxes):
    x0, y0 = min(b[0] for b in boxes), min(b[1] for b in boxes)
    return (x0, y0, max(b[0] + b[2] for b in boxes) - x0, max(b[1] + b[3] for b in boxes) - y0)


FORMATS = {"u8": (None, 1, True), "f32": (tensor_format("float32", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True), 4, False),
           "u8hwc": (tensor_format("uint8", "hwc"), 1, True), "bf16": (tensor_format("bfloat16", "hwc", "mul", drop_alpha=True), 2, False)}


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("ep", ENTRY_POINTS)
def test_shared_equals_per_entry(codec, ep, level):
    """Interleaved entries (a, b, a, c, b, a, ...) of an RGB file with 30 entries, an RGBA file with 8 and an RGB file with
    one, every op and a mix of colour, blur and augment entries: the call with each file packed once gives the bytes of the
    call with each entry's file at its own offset, and decodes each file's tile bounding box once."""
    rng = np.random.default_rng(ENTRY_POINTS.index(ep) * 3 + level)
    imgs = [synth.rgb(700, 900, 10 + level), synth.rgba(300, 1000, 11 + level), synth.rgb(150, 200, 12 + level)]
    files = [po.encode(level, im) for im in imgs]
    heads = [(im.shape[1], im.shape[0], im.shape[2] == 4) for im in imgs]
    idx = interleaved(rng)
    entry_files = [files[k] for k in idx]
    fmts = ["u8"] if ep in ("region", "oriented", "resized") else ["u8hwc", "f32", "bf16"] if ep == "tensor" else ["u8", "f32"]
    for fk in fmts:
        fmt, eb, alpha_kept = FORMATS[fk]
        e = entries(rng, idx, heads, alpha_kept)
        nb = []
        for j, k in enumerate(idx):
            h, w = out_hw(ep, e, j, None)
            c = 3 + heads[k][2] if fmt is None or fmt.channels == 0 else 3
            nb.append(h * w * c * eb)
        want, t_own = run(codec, ep, entry_files, e, nb, fmt, share=False)
        got, t_shared = run(codec, ep, entry_files, e, nb, fmt, share=True)
        assert got.tobytes() == want.tobytes(), (ep, level, fk)
        if level == 7:
            assert t_own == t_shared == 0
            continue
        if ep in ("region", "oriented", "resized", "tensor"):   # the decoded rectangle is the box (a resize reads all of it)
            per_entry = sum(region_tiles(heads[k][0], heads[k][1], e["boxes"][j])[0] for j, k in enumerate(idx))
            once = sum(region_tiles(heads[k][0], heads[k][1], bbox([e["boxes"][j] for j, kk in enumerate(idx) if kk == k]))[0]
                       for k in range(3))
            assert (t_own, t_shared) == (per_entry, once), (ep, fk)
        assert t_shared < t_own


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_dino_views_one_call(codec, level):
    """DINO's 2 global + 6 local views of a batch through one decode_views call, under the seeds and draws of
    test_blur_decode.test_dino_views_replayed: bit-identical to DINO's PIL Compose, and each file's tiles decoded once."""
    import torch
    import torchvision.transforms as T
    from torchvision.transforms import InterpolationMode as IM
    imgs = [synth.rgb(h, w, 1900 + k) for k, (w, h) in enumerate([(500, 375), (333, 500), (640, 427), (300, 300)] * 3)]
    files = [po.encode(level, im) for im in imgs]
    cj = T.ColorJitter(0.4, 0.4, 0.2, 0.1)
    flip_and_color = T.Compose([T.RandomHorizontalFlip(p=0.5), T.RandomApply([cj], p=0.8), T.RandomGrayscale(p=0.2)])
    normalize = T.Compose([T.ToTensor(), T.Normalize(*IMAGENET.values())])
    g1 = T.RandomResizedCrop(224, scale=(0.4, 1.0), interpolation=IM.BICUBIC)
    g2 = T.RandomResizedCrop(224, scale=(0.4, 1.0), interpolation=IM.BICUBIC)
    lc = T.RandomResizedCrop(96, scale=(0.05, 0.4), interpolation=IM.BICUBIC)
    views = [(g1, T.Compose([g1, flip_and_color, DinoGaussianBlur(1.0), normalize]), 1.0, 0.0),
             (g2, T.Compose([g2, flip_and_color, DinoGaussianBlur(0.1), DinoSolarization(0.2), normalize]), 0.1, 0.2)]
    views += [(lc, T.Compose([lc, flip_and_color, DinoGaussianBlur(p=0.5), normalize]), 0.5, 0.0)] * 6
    torch.manual_seed(82 + level)
    random.seed(82 + level)
    want = [[tf(Image.fromarray(im)) for _, tf, _, _ in views] for im in imgs]
    torch.manual_seed(82 + level)
    random.seed(82 + level)
    draws = [[_replay_view(rrc, Image.fromarray(im), cj, bp, sp) for rrc, _, bp, sp in views] for im in imgs]
    args = []
    for v, (rrc, _, _, _) in enumerate(views):
        d = [dr[v] for dr in draws]
        s = rrc.size[0]
        args.append(dict(sizes=[(s, s)] * len(files), boxes=[x[0] for x in d], ops=[x[1] for x in d], filters="bicubic",
                         colors=[x[2] for x in d], blurs=[x[3] for x in d]))
    got = codec.decode_views(files, args, torch.float32, mean=IMAGENET["mean"], std=IMAGENET["std"])
    assert len(got) == len(views)
    for v, g in enumerate(got):
        assert g.shape == (len(files), 3, views[v][0].size[0], views[v][0].size[0])
        assert torch.equal(g.cpu().view(torch.int32), torch.stack([w[v] for w in want]).view(torch.int32)), v
    once = sum(region_tiles(im.shape[1], im.shape[0], bbox([dr[v][0] for v in range(len(views))]))[0] for im, dr in zip(imgs, draws))
    per_view = sum(region_tiles(im.shape[1], im.shape[0], dr[v][0])[0] for im, dr in zip(imgs, draws) for v in range(len(views)))
    assert codec.last_tiles == once < per_view


@gpu
@pytest.mark.parametrize("family", ("batch", "latency"))
def test_pipelined_shared_chunks(monkeypatch, family):
    """Interleaved repeats of sintel-like frames cut into at least 3 chunks on 2 lanes: host buffers (each chunk copies back
    only its own entries, which other chunks' entries sit between) and device buffers, uint8 and float32, through the batch
    and the latency kernel families: the bytes of the per-entry call."""
    frames = synth.sintel_batch(range(3100, 3105))
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "2")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "2")
    if family == "batch":
        monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(311)
        idx = [int(k) for k in rng.integers(0, len(frames), 24)] + list(range(len(frames)))
        heads = [(f.shape[1], f.shape[0], False) for f in frames]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            entry_files = [files[k] for k in idx]
            e = entries(rng, idx, heads, False)
            e["boxes"] = [(int(rng.integers(0, 900)), int(rng.integers(0, 500)), int(rng.integers(200, 1000)), int(rng.integers(100, 500)))
                          for _ in idx]
            e["szs"] = [(224, 224) if j % 2 else (b[2], b[3]) for j, b in enumerate(e["boxes"])]
            e["wins"] = [(0, 0, z[0], z[1]) for z in e["szs"]]
            e["augs"] = [None] * len(idx)
            for fmt, eb in ((None, 1), (FORMATS["f32"][0], 4)):
                nb = [out_hw("blur", e, j, None)[0] * out_hw("blur", e, j, None)[1] * 3 * eb for j in range(len(idx))]
                for dev in (False, True):
                    want, t_own = run(cd, "blur", entry_files, e, nb, fmt, share=False, dev=dev)
                    cd.profile(True)
                    got, t_shared = run(cd, "blur", entry_files, e, nb, fmt, share=True, dev=dev)
                    rep = cd.profile_report()
                    cd.profile(False)
                    assert rep["k_dec_tile_offsets"][1] >= 3, rep   # one launch per chunk
                    assert got.tobytes() == want.tobytes(), (lv, fmt is None, dev)
                    assert t_shared < t_own
    finally:
        cd.close()


@gpu
def test_shared_failures(codec, monkeypatch):
    """A refused entry of a shared file is named by the caller's index; a corrupt shared file fails the call, and the call
    returns only once every chunk it issued has finished (the output is quiet, and the context decodes on)."""
    import torch
    a, b = po.encode(1, synth.rgb(500, 600, 21)), po.encode(2, synth.rgba(200, 300, 22))
    files = [a, b, a, a, b, a]
    boxes = [(0, 0, 100, 100), (5, 5, 50, 50), (100, 100, 300, 300), (550, 0, 60, 10), (0, 0, 300, 200), (1, 1, 1, 1)]
    nb = [bx[2] * bx[3] * 4 for bx in boxes]
    descs, foffs, fsizes, fb, poff = pack(files, nb, share=True)
    out = np.full(poff + 16, 0xA5, np.uint8)
    fa = np.frombuffer(fb, np.uint8)
    with pytest.raises(RuntimeError, match=r"entry 3: rectangle \(550, 0\) 60x10 is not inside the 600x500 image"):
        codec.decode_region_raw(descs, rects(boxes), len(files), fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
    assert (out == 0xA5).all()
    ops = ["tl", "tl", "tl", "r90", "tl", "tl"]
    bad_ops = op_codes(ops)
    bad_ops[4] = 99
    with pytest.raises(RuntimeError, match="entry 4: unknown orientation op 99"):
        codec.decode_oriented_raw(descs, bad_ops, rects([(0, 0, 10, 10)] * 6), 6, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                  out.ctypes.data, poff, 0)
    assert (out == 0xA5).all()
    # corrupt the first tile's size field of the shared level-1 file, in a call cut into several chunks
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "2")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "1")
    cd = xpng_b200.Codec(0)
    try:
        frames = [synth.rgb(1000, 1200, 30 + k) for k in range(4)]
        good = cd.encode(1, frames)
        bad = bytearray(good[1])
        bad[9] ^= 0xFF; bad[10] ^= 0x7F
        bad = bytes(bad)
        fs = [good[0], bad, good[2], bad, good[3], bad, good[0]]
        bxs = [(0, 0, 1200, 1000)] * len(fs)
        nb = [1200 * 1000 * 3] * len(fs)
        descs, foffs, fsizes, fb, poff = pack(fs, nb, share=True)
        dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
        dout = torch.zeros(poff + 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with pytest.raises(RuntimeError, match="corrupt"):
            cd.decode_region_raw(descs, rects(bxs), len(fs), dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dout.data_ptr(), poff, 1)
        first = dout.cpu()
        torch.cuda._sleep(50_000_000)   # anything still in flight would land during this
        torch.cuda.synchronize()
        assert torch.equal(first, dout.cpu())
        for j in (0, 2, 4, 6):   # chunks without the corrupt file were issued and finished
            got = first[descs[j].offset: descs[j].offset + nb[j]].numpy().reshape(1000, 1200, 3)
            assert np.array_equal(got, frames[[0, 0, 2, 2, 3, 3, 0][j]]) or not got.any(), j
        assert all(np.array_equal(x, f) for x, f in zip(cd.decode_region(good, [(0, 0, 1200, 1000)] * 4), frames))
    finally:
        cd.close()
