"""Tensor decode (xpngb_decode_tensor / Codec.decode_tensor): each decoded, cropped, resized or turned entry written as a
normalised tensor, bit-identical to torchvision's to_tensor / ToDtype(scale=True) followed by Normalize.

to_tensor_ref() restates the arithmetic contract of include/xpng_b200.h in numpy float32.  Without a GPU it is pinned to
torchvision on all 256 byte values.  On the GPU every output equals to_tensor_ref of what decode_resized / decode_oriented /
decode_region write for the entry, and a sample of RandomResizedCrop-style entries equals torchvision's own pipelines.
Every comparison is on bit patterns, so -0.0 and the last ulp count."""
import ctypes as C
import hashlib

import numpy as np
import pytest
import torch
from PIL import Image

from conftest import make_case, manifest
from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import DTYPE_BYTES, op_codes, rects, sizes as size_arr, tensor_format
from test_region import GENS, grid_rects, halfflat
from test_resized_decode import pack, resize_bilinear, rrc_boxes, size_kinds

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
IMAGENET = dict(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
IMAGENET4 = dict(mean=(0.485, 0.456, 0.406, 0.5), std=(0.229, 0.224, 0.225, 0.25))
DTYPES = ("uint8", "float32", "float16", "bfloat16")
BITS = {"uint8": np.uint8, "float32": np.uint32, "float16": np.uint16, "bfloat16": np.uint16}


# ---------------------------------------------------------------------------------------------------- the reference

def _bf16_bits(y):
    """float32 -> bfloat16 bit patterns, round to nearest even (finite inputs)."""
    u = y.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def to_tensor_ref(px, dtype="float32", layout="chw", scale="div", mean=(0, 0, 0, 0), std=(1, 1, 1, 1), drop_alpha=False):
    """The (h, w, c) uint8 array px as xpngb_decode_tensor writes it, as bit patterns (BITS[dtype]): (C, h, w) or (h, w, C)."""
    if drop_alpha:
        px = px[:, :, :3]
    c = px.shape[2]
    if dtype == "uint8":
        t = px
    else:
        b = px.astype(np.float32)
        v = b / np.float32(255) if scale == "div" else b * np.float32(1.0 / 255)
        m = np.array((list(mean) + [0.0] * 4)[:c], np.float32)
        s = np.array((list(std) + [1.0] * 4)[:c], np.float32)
        y = ((v - m) / s).astype(np.float32)
        t = {"float32": lambda: y.view(np.uint32), "float16": lambda: y.astype(np.float16).view(np.uint16),
             "bfloat16": lambda: _bf16_bits(y)}[dtype]()
    return np.ascontiguousarray(t.transpose(2, 0, 1) if layout == "chw" else t)


def bits(t):
    """A torch tensor's bit patterns as numpy."""
    t = t.detach().cpu()
    return {torch.float32: lambda: t.view(torch.int32).numpy().view(np.uint32), torch.float16: lambda: t.view(torch.int16).numpy().view(np.uint16),
            torch.bfloat16: lambda: t.view(torch.int16).numpy().view(np.uint16), torch.uint8: lambda: t.numpy()}[t.dtype]()


# ---------------------------------------------------------------------------------------------------- reference against torchvision (CPU)

def _all_bytes(c):
    """A 16 x 16 image whose every channel holds each byte value once (channels rotated against each other)."""
    v = np.arange(256, dtype=np.uint8)
    return np.stack([np.roll(v, 37 * k) for k in range(c)], axis=1).reshape(16, 16, c)


@pytest.mark.parametrize("mode", ("RGB", "RGBA"))
def test_reference_matches_torchvision(mode):
    import torchvision.transforms.functional as F
    from torchvision.transforms import v2
    px = _all_bytes(len(mode))
    pil = Image.fromarray(px, mode)
    norms = [IMAGENET if mode == "RGB" else IMAGENET4, dict(mean=(0, 0, 0, 0)[:len(mode)], std=(1, 1, 1, 1)[:len(mode)])]
    for nm in norms:
        mean, std = list(nm["mean"]), list(nm["std"])
        v1 = F.normalize(F.to_tensor(pil), mean, std)
        v2t = v2.Normalize(mean, std)(v2.ToDtype(torch.float32, scale=True)(v2.ToImage()(pil)))
        for dt in ("float32", "float16", "bfloat16"):
            tdt = getattr(torch, dt)
            assert np.array_equal(to_tensor_ref(px, dt, "chw", "div", mean, std), bits(v1.to(tdt))), (nm, dt)
            assert np.array_equal(to_tensor_ref(px, dt, "chw", "mul", mean, std), bits(v2t.to(tdt))), (nm, dt)
            assert np.array_equal(to_tensor_ref(px, dt, "hwc", "div", mean, std), bits(v1.to(tdt).permute(1, 2, 0).contiguous()))
        if not any(mean) and all(s == 1 for s in std):   # mean 0 / std 1 is the pipeline without Normalize
            assert np.array_equal(to_tensor_ref(px, "float32", "chw", "div", mean, std), bits(F.to_tensor(pil)))
            assert np.array_equal(to_tensor_ref(px, "float32", "chw", "mul", mean, std),
                                  bits(v2.ToDtype(torch.float32, scale=True)(v2.ToImage()(pil))))
    assert np.array_equal(to_tensor_ref(px, "uint8", "chw"), F.pil_to_tensor(pil).numpy())
    assert np.array_equal(to_tensor_ref(px, "uint8", "chw"), v2.ToImage()(pil).numpy())
    if mode == "RGBA":
        assert np.array_equal(to_tensor_ref(px, "float32", drop_alpha=True), bits(F.to_tensor(pil.convert("RGB"))))


def test_div_and_mul_scales_differ():
    """x / 255 and x * float32(1 / 255) disagree on 126 of the 256 byte values: the two modes must stay distinct."""
    px = np.arange(256, dtype=np.uint8).reshape(1, 256, 1).repeat(3, axis=2)
    d, m = to_tensor_ref(px, scale="div"), to_tensor_ref(px, scale="mul")
    assert int((d[0] != m[0]).sum()) == 126


def test_tensor_format_fields():
    f = tensor_format(torch.bfloat16, "hwc", "mul", IMAGENET["mean"], IMAGENET["std"], drop_alpha=True)
    assert (f.dtype, f.layout, f.scale, f.channels) == (3, 1, 1, 3)
    assert list(f.mean) == [np.float32(v) for v in IMAGENET["mean"]] + [0.0] and list(f.std)[3] == 1.0
    assert tensor_format("uint8").dtype == 0 and tensor_format(torch.float16).channels == 0
    for bad in (dict(dtype=torch.int32), dict(dtype="float32", layout="nchw"), dict(dtype="float32", scale="x")):
        with pytest.raises(ValueError):
            tensor_format(**bad)


# ---------------------------------------------------------------------------------------------------- tensor decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def pixels_of(full, rect=None, size=None, op=None):
    """What decode_resized / decode_oriented / decode_region write for the entry (uint8 HWC)."""
    if rect is not None:
        x, y, w, h = rect
        full = full[y: y + h, x: x + w]
    if size is not None:
        full = resize_bilinear(full, *size)
    return po.orient(op or "tl", full)


def out_shape(hdr_wh, a, fmt, rect=None, size=None, op=None):
    w, h = size if size is not None else (rect[2], rect[3]) if rect is not None else hdr_wh
    if op in ("r90", "r270"):
        w, h = h, w
    c = 3 if fmt.get("drop_alpha") else 3 + a
    return (c, h, w) if fmt.get("layout", "chw") == "chw" else (h, w, c)


SENTINEL = 0xA5


def run(cd, files, fmt, boxes=None, szs=None, ops=None, files_dev=False, out_dev=True):
    """xpngb_decode_tensor into a sentinel-filled buffer with 16 guard bytes after every entry; returns the entries as bit
    pattern arrays after checking that no byte outside them changed.  With host output a call copies each chunk's span of
    entries back in one piece (the gaps between entries included, as for every decode call), so there only the bytes past
    the last entry are checked."""
    dt = fmt.get("dtype", "float32")
    eb = DTYPE_BYTES[dt]
    hdrs = [po.decode(f).shape for f in files]
    shapes = [out_shape((s[1], s[0]), int(s[2] == 4), fmt, None if boxes is None else boxes[i], None if szs is None else szs[i],
                        None if ops is None else ops[i]) for i, s in enumerate(hdrs)]
    nbytes = [int(np.prod(s)) * eb + 16 for s in shapes]                      # 16 guard bytes after each entry
    descs, foffs, fsizes, fb, poff = pack(files, nbytes)
    cap = poff + 64
    if out_dev:
        out = torch.full((cap,), SENTINEL, dtype=torch.uint8, device="cuda")
        optr = out.data_ptr()
    else:
        out = np.full(cap, SENTINEL, np.uint8)
        optr = out.ctypes.data
    fa = np.frombuffer(fb, np.uint8)
    if files_dev:
        dfiles = torch.from_numpy(fa.copy()).cuda()
        fptr = dfiles.data_ptr()
    else:
        fptr = fa.ctypes.data
    torch.cuda.synchronize()
    cd.decode_tensor_raw(tensor_format(dt, fmt.get("layout", "chw"), fmt.get("scale", "div"), fmt.get("mean", (0, 0, 0, 0)),
                                       fmt.get("std", (1, 1, 1, 1)), fmt.get("drop_alpha", False)),
                         descs, None if ops is None else op_codes(ops), None if boxes is None else rects(boxes),
                         None if szs is None else size_arr(szs), len(files), fptr, len(fb), int(files_dev), foffs, fsizes, optr, cap,
                         int(out_dev))
    host = out.cpu().numpy() if out_dev else out
    written = np.zeros(cap, bool)
    got = []
    for i, s in enumerate(shapes):
        a, b = descs[i].offset, descs[i].offset + int(np.prod(s)) * eb
        written[a:b] = True
        got.append(host[a:b].view(BITS[dt]).reshape(s))
    if not out_dev:
        written[:max(descs[i].offset + int(np.prod(s)) * eb for i, s in enumerate(shapes))] = True
    assert (host[~written] == SENTINEL).all(), "bytes outside the entries changed"
    return got


def check(cd, files, fmt, boxes=None, szs=None, ops=None, **kw):
    got = run(cd, files, fmt, boxes, szs, ops, **kw)
    fulls = {}
    for i, (f, g) in enumerate(zip(files, got)):
        if f not in fulls:
            fulls[f] = po.decode(f)
        px = pixels_of(fulls[f], None if boxes is None else boxes[i], None if szs is None else szs[i], None if ops is None else ops[i])
        want = to_tensor_ref(px, **fmt)
        assert g.shape == want.shape and np.array_equal(g, want), (i, fmt, None if boxes is None else boxes[i],
                                                                    None if szs is None else szs[i], None if ops is None else ops[i])
    return got


F32_IMAGENET = dict(dtype="float32", layout="chw", scale="div", **IMAGENET)


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("gen", sorted(GENS))
def test_tensor_against_reference(codec, gen, level):
    rng = np.random.default_rng(sorted(GENS).index(gen) * 3 + level + 300)
    h, w = 700, 1000                         # 2 x 2 tiles, as test_region_against_oracle
    f = po.encode(level, GENS[gen](h, w, 46))
    boxes = grid_rects(w, h, rng)
    entries = [(r, op) for r in boxes for op in ALL_OPS]
    check(codec, [f] * len(entries), F32_IMAGENET, [r for r, _ in entries], None, [op for _, op in entries])
    check(codec, [f] * len(ALL_OPS), F32_IMAGENET, None, None, ALL_OPS)      # whole images, every op
    check(codec, [f], F32_IMAGENET)                                          # whole image, no op


def _formats():
    out = []
    for dt in DTYPES:
        for layout in ("chw", "hwc"):
            for scale in ("div", "mul"):
                for drop in (False, True):
                    out.append(dict(dtype=dt, layout=layout, scale=scale, drop_alpha=drop, **IMAGENET4))
    return out


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_tensor_format_matrix(codec, level):
    imgs = [synth.rgba(500, 460, 71), synth.rgb(300, 520, 72), halfflat(460, 700, 73)]
    files = [po.encode(level, im) for im in imgs] + [po.encode(7, imgs[0])]
    batch, boxes, szs, ops = [], [], [], []
    for k, (f, im) in enumerate(zip(files, imgs + imgs[:1])):
        h, w = im.shape[:2]
        for r, z, op in (((0, 0, w, h), None, ALL_OPS[k]), ((17, 9, w - 40, h - 31), None, "r90"), ((3, 5, 101, 77), (224, 224), "mh"),
                         ((w // 2, 1, w // 2, h - 1), (31, 64), "r270")):
            batch.append(f); boxes.append(r); szs.append(z if z is not None else (r[2], r[3])); ops.append(op)
    for fmt in _formats():
        check(codec, batch, fmt, boxes, szs, ops)
        check(codec, batch[:4], fmt, None, None, ops[:4])


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_tensor_resized(codec, level):
    rng = np.random.default_rng(level + 500)
    for gen in ("rgb", "rgba"):
        h, w = 700, 1000
        f = po.encode(level, GENS[gen](h, w, 47))
        boxes = grid_rects(w, h, rng)
        entries = [(r, z) for r in boxes for z in size_kinds(r[2], r[3])]
        ops = [ALL_OPS[k % len(ALL_OPS)] for k in range(len(entries))]
        check(codec, [f] * len(entries), F32_IMAGENET, [r for r, _ in entries], [z for _, z in entries], ops)
        check(codec, [f] * 6, dict(dtype="bfloat16", layout="hwc", scale="mul", **IMAGENET4), None, size_kinds(w, h), None)


@gpu
def test_tensor_matches_torchvision_pipelines(codec):
    """RandomResizedCrop(224) + RandomHorizontalFlip + ToTensor + Normalize, in torchvision v1 and v2, against one call."""
    import torchvision.transforms.functional as F
    from torchvision.transforms import v2
    from torchvision.transforms import InterpolationMode
    frames = synth.sintel_batch(range(1000, 1012))
    rng = np.random.default_rng(2029)
    boxes = rrc_boxes(rng, len(frames))
    ops = [("mh", "tl")[int(rng.integers(2))] for _ in frames]
    assert 0 < ops.count("mh") < len(ops)
    for lv in (1, 2):
        files = codec.encode(lv, frames)
        pils = [Image.fromarray(po.decode(f)) for f in files]
        crops = []
        for p, (x, y, w, h), op in zip(pils, boxes, ops):
            c = F.resized_crop(p, y, x, h, w, [224, 224], InterpolationMode.BILINEAR)
            crops.append(F.hflip(c) if op == "mh" else c)
        mean, std = list(IMAGENET["mean"]), list(IMAGENET["std"])
        v1 = torch.stack([F.normalize(F.to_tensor(c), mean, std) for c in crops])
        got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, scale="div", **IMAGENET)
        assert got.shape == (len(files), 3, 224, 224) and np.array_equal(bits(got), bits(v1))
        v2p = v2.Compose([v2.ToImage(), v2.ToDtype(torch.float32, scale=True), v2.Normalize(mean, std)])
        v2t = torch.stack([v2p(c) for c in crops])
        for dt in (torch.float32, torch.bfloat16):
            got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, dtype=dt, scale="mul", **IMAGENET)
            assert got.dtype == dt and np.array_equal(bits(got), bits(v2t.to(dt))), dt


@gpu
def test_u8_hwc_is_the_pixel_decode(codec):
    imgs = [synth.rgb(700, 1000, 31), synth.rgba(500, 460, 32), synth.rgb(1, 999, 33), synth.rgba(333, 129, 34)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7, 7), imgs)]
    rng = np.random.default_rng(5)
    boxes = [grid_rects(im.shape[1], im.shape[0], rng)[-4] for im in imgs]
    szs = [(224, 224), (100, 33), (1, 5), (64, 200)]
    ops = ["r90", "mh", "r270", "mvh"]
    u8 = dict(dtype="uint8", layout="hwc")

    def same(a, b):
        assert len(a) == len(b) and all(x.shape == y.shape and x.tobytes() == y.tobytes() for x, y in zip(a, b))

    same(run(codec, files, u8, boxes, szs, ops), codec.decode_resized(files, szs, boxes, ops))
    same(run(codec, files, u8, None, szs, None), codec.decode_resized(files, szs))
    same(run(codec, files, u8, boxes, None, ops), codec.decode_region(files, boxes, ops))
    same(run(codec, files, u8, boxes), codec.decode_region(files, boxes))
    same(run(codec, files, u8, None, None, ops), codec.decode(files, ops))
    same(run(codec, files, u8), codec.decode(files))


def _lut(fmt, c):
    """Bit patterns of the 256 byte values in channel c under fmt (the contract is per byte and channel)."""
    px = np.zeros((1, 256, 4), np.uint8)
    px[0, :, c] = np.arange(256)
    return to_tensor_ref(px, **{**fmt, "layout": "hwc", "drop_alpha": False})[0, :, c]


@gpu
@pytest.mark.parametrize("name", ("rgb_4k_s1", "rgba_8192_s2"))
def test_tensor_large_golden(codec, name):
    entry = manifest()["synthetic"][name]
    px = make_case("synthetic", name, entry)
    f = codec.encode(1, [px])[0]
    assert hashlib.sha256(f).hexdigest() == entry["levels"]["1"]["sha256"]
    ref = po.decode(f)
    for drop in (False, True):
        fmt = dict(dtype="float16", layout="chw", scale="div", **IMAGENET4)
        got = codec.decode_tensor([f], dtype=torch.float16, drop_alpha=drop, **IMAGENET4)
        c = 3 if drop else ref.shape[2]
        assert got.shape == (1, c, ref.shape[0], ref.shape[1])
        g = bits(got[0])
        for k in range(c):
            assert np.array_equal(g[k], _lut(fmt, k)[ref[:, :, k]]), (name, drop, k)
        del got, g


@gpu
def test_tensor_batch_kernel_family(monkeypatch):
    """The pair decoders, three-tile walk and row-pitched un-predict (selected by batch size), forced on small inputs."""
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(9)
        for lv in (1, 2):
            for im in (synth.rgb(700, 1000, 91), synth.rgba(900, 700, 92), halfflat(700, 1000, 24)):
                h, w = im.shape[:2]
                f = po.encode(lv, im)
                boxes = grid_rects(w, h, rng)
                szs = [size_kinds(r[2], r[3])[k % 6] for k, r in enumerate(boxes)]
                ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in boxes]
                check(cd, [f] * len(boxes), F32_IMAGENET, boxes, szs, ops)
                check(cd, [f] * len(boxes), dict(dtype="float16", layout="hwc", scale="mul", **IMAGENET4), boxes, None, ops)
    finally:
        cd.close()


@gpu
def test_tensor_pipelined_chunks_and_profile(monkeypatch):
    """24 sintel-like frames in 1 MPix chunks on two lanes (every lane reused), through the batch kernel family; the profile
    shows one k_to_tensor launch per chunk and no crop or orientation launch."""
    frames = synth.sintel_batch(range(1000, 1024))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "2")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(67)
        boxes = rrc_boxes(rng, len(frames))
        ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in frames]
        files = cd.encode(1, frames)
        for profiled in (True, False):
            cd.profile(profiled)
            check(cd, files, F32_IMAGENET, boxes, [(224, 224)] * len(files), ops)
            check(cd, files[:6], dict(dtype="bfloat16", layout="chw", scale="mul", **IMAGENET), boxes[:6], None, ops[:6])
            if profiled:
                rep = cd.profile_report()
                assert rep["k_to_tensor"][1] == rep["k_dec_parse_m1"][1] >= 3, rep
                assert "k_orient" not in rep and "k_crop_rows" not in rep, sorted(rep)
    finally:
        cd.close()


@gpu
def test_tensor_profile_single_chunk(codec):
    f = po.encode(2, synth.rgb(700, 1000, 12))
    codec.profile(True)
    try:
        check(codec, [f] * 3, F32_IMAGENET, [(0, 0, 1000, 700), (0, 0, 588, 636), (5, 5, 50, 50)], None, ["tl", "r90", "mh"])
        rep = codec.profile_report()
    finally:
        codec.profile(False)
    assert rep["k_to_tensor"][1] == 1 and "k_orient" not in rep and "k_crop_rows" not in rep, rep


@gpu
def test_tensor_device_and_host_buffers(codec):
    frames = [synth.rgb(720, 1280, 60), synth.rgba(600, 900, 61), synth.rgb(333, 517, 62), synth.rgba(64, 48, 63)]
    files = [po.encode(lv, f) for lv, f in zip((1, 1, 2, 7), frames)]
    boxes = [(100, 37, 600, 500), (0, 444, 900, 156), (17, 3, 1, 300), (3, 5, 41, 29)]
    szs = [(224, 224), (100, 333), (517, 1), (96, 80)]
    fmt = dict(dtype="float16", layout="chw", scale="div", **IMAGENET4)
    for files_dev, out_dev in ((True, True), (False, True), (True, False), (False, False)):
        for ops in (["r90", "mh", "r270", "mv"], None):
            check(codec, files, fmt, boxes, szs, ops, files_dev=files_dev, out_dev=out_dev)
            check(codec, files, fmt, None, None, ops, files_dev=files_dev, out_dev=out_dev)


@gpu
def test_tensor_failures(codec):
    px = synth.rgb(600, 700, 5)
    f = po.encode(1, px)
    good = tensor_format("float32", **IMAGENET)

    def call(fmt, files=(f, f), szs=None, boxes=None, offset=None, fmt_null=False):
        descs, foffs, fsizes, fb, poff = pack(list(files), [700 * 600 * 4 * 4] * len(files))
        if offset is not None:
            descs[len(files) - 1].offset = offset
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, SENTINEL, np.uint8)
        rc = xpng_b200.lib().xpngb_decode_tensor(codec._h, None if fmt_null else C.byref(fmt), None, descs,
                                                 None if boxes is None else rects(boxes), None if szs is None else size_arr(szs),
                                                 len(files), fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
        return rc, codec._err(), (out == SENTINEL).all()

    def bad(**changes):
        fmt = tensor_format("float32", **IMAGENET)
        for k, v in changes.items():
            if isinstance(v, tuple):
                getattr(fmt, k)[v[0]] = v[1]
            else:
                setattr(fmt, k, v)
        return fmt

    rc, err, untouched = call(good, fmt_null=True)
    assert rc == 1 and "fmt" in err and untouched
    for fmt, word in ((bad(dtype=4), "dtype"), (bad(layout=2), "layout"), (bad(scale=7), "scale"), (bad(channels=1), "channels"),
                      (bad(channels=4), "channels"), (bad(std=(1, 0.0)), "std[1]"), (bad(std=(2, float("nan"))), "std[2]"),
                      (bad(std=(0, float("inf"))), "std[0]"), (bad(mean=(2, float("nan"))), "mean[2]"),
                      (bad(channels=0, std=(3, 0.0)), "std[3]"), (bad(mean=(0, float("-inf"))), "mean[0]")):
        rc, err, untouched = call(fmt)
        assert rc == 1 and word in err and untouched, (word, err)
    # a channel that is not used is not checked: alpha dropped, or a uint8 tensor
    assert call(bad(channels=3, std=(3, 0.0)))[0] == 0
    assert call(bad(dtype=0, std=(0, float("nan"))))[0] == 0
    descs, foffs, fsizes, fb, poff = pack([f], [600 * 700 * 3 * 4])
    fa = np.frombuffer(fb, np.uint8)
    out = np.full(poff + 64, SENTINEL, np.uint8)
    rc = xpng_b200.lib().xpngb_decode_tensor(codec._h, C.byref(good), None, descs, None, None, 1, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                             out.ctypes.data, 600 * 700 * 3 * 4 - 1, 0)   # the tensor one byte past out_cap
    assert rc == 1 and "exceed" in codec._err() and (out == SENTINEL).all()
    rc, err, untouched = call(good, offset=600 * 700 * 3 * 4 + 8)           # misaligned output offset
    assert rc == 1 and "file 1" in err and "multiple of 16" in err and untouched
    rc, err, untouched = call(good, boxes=[(0, 0, 5, 5), (0, 0, 701, 10)])    # a rectangle not inside its image
    assert rc == 1 and "entry 1" in err and untouched
    rc, err, untouched = call(good, szs=[(5, 5), (0, 3)])
    assert rc == 1 and "entry 1" in err and untouched
    # and the context still decodes afterwards
    check(codec, [f], F32_IMAGENET, None, None, ["mh"])


@gpu
def test_codec_decode_tensor(codec):
    imgs = [synth.rgb(300, 500, 1), synth.rgba(300, 500, 2), synth.gray_as_rgb(500, 300, 3)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)]
    got = codec.decode_tensor(files, [(56, 56)] * 3, None, ["tl", "mh", "r90"], drop_alpha=True, **IMAGENET)
    assert got.shape == (3, 3, 56, 56) and got.dtype == torch.float32 and got.device == torch.device("cuda", codec.device)
    raw = run(codec, files, dict(drop_alpha=True, **F32_IMAGENET), None, [(56, 56)] * 3, ["tl", "mh", "r90"])
    assert np.array_equal(bits(got), np.stack(raw))
    # odd element counts: entries sit at 16-byte offsets inside, the returned batch is contiguous
    got = codec.decode_tensor(files[:1] * 3, [(5, 7)] * 3, dtype=torch.float16, layout="hwc")
    assert got.shape == (3, 7, 5, 3) and got.is_contiguous()
    assert np.array_equal(bits(got), np.stack(run(codec, files[:1] * 3, dict(dtype="float16", layout="hwc"), None, [(5, 7)] * 3)))
    u8 = codec.decode_tensor(files[:1], boxes=[(10, 20, 30, 40)], dtype=torch.uint8)
    assert u8.shape == (1, 3, 40, 30) and np.array_equal(u8[0].cpu().numpy(), po.decode(files[0])[20:60, 10:40].transpose(2, 0, 1))
    for kw in (dict(sizes=[(64, 48), (48, 64), (64, 48)]),                   # mixed sizes
               dict(sizes=[(64, 48)] * 3, drop_alpha=False),                 # mixed alpha
               dict(sizes=[(64, 48)] * 3, ops=["tl", "r90", "tl"], drop_alpha=True)):   # a quarter turn of a non-square output
        with pytest.raises(ValueError, match="shapes"):
            codec.decode_tensor(files, **kw)
    with pytest.raises(RuntimeError, match="entry 1"):
        codec.decode_tensor(files[:2], boxes=[(0, 0, 5, 5), (498, 0, 5, 5)], drop_alpha=True)
