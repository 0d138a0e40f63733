"""Colour decode (xpngb_decode_color / Codec.decode_resized and decode_tensor with colors): torchvision's ColorJitter and
RandomGrayscale applied to each entry, byte-identical to their PIL path.  Entry i is
tensor(gray_i(jitter_i(orient(op_i, window_i(resize_f(crop_i)))))).

color_ref() restates the steps in numpy, operation for operation as Pillow rounds them (Blend.c, Convert.c, ImageStat).  The
CPU tests pin it to the installed Pillow and torchvision: each step alone, the HSV round trip over all 2^24 inputs, and a
seeded ColorJitter + RandomGrayscale.  On the GPU every output is compared with color_ref of po.decode's pixels."""
import ctypes as C
import math

import numpy as np
import pytest
from PIL import Image

from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import _Color, color_array, color_params, filter_codes, op_codes, rects, sizes as size_arr, tensor_format
from test_resampled_decode import FILTERS, pack, resize_pil, window
from test_tensor_decode import IMAGENET, bits, to_tensor_ref

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
F32, F64 = np.float32, np.float64


# ---------------------------------------------------------------------------------------------------- the oracle

def luma(px):
    """Pillow's L24 luma of an (..., >= 3) uint8 array, as int64."""
    p = px.astype(np.int64)
    return (19595 * p[..., 0] + 38470 * p[..., 1] + 7471 * p[..., 2] + 0x8000) >> 16


def blend(d, p, f):
    """Image.blend(deg, img, f) of one channel: float32 arithmetic, each operation rounded, truncated and clipped."""
    a = F32(f)
    t = np.asarray(d).astype(F32) + a * (p.astype(np.int64) - d).astype(F32)
    return np.where(t <= 0, 0, np.where(t >= 255, 255, np.clip(t, 0, 255).astype(np.int64))).astype(np.uint8)


def _round(x):
    """C's round of non-negative doubles: half away from zero (numpy's round is half to even)."""
    t = np.trunc(x)
    return (t + (x - t >= 0.5)).astype(np.int64)


def rgb2hsv(px):
    """Pillow's rgb2hsv (Convert.c) of an (..., 3) uint8 array -> H, S, V as int64 arrays."""
    r, g, b = (px[..., k].astype(np.int64) for k in range(3))
    mx, mn = np.maximum(r, np.maximum(g, b)), np.minimum(r, np.minimum(g, b))
    grey = mx == mn
    with np.errstate(divide="ignore", invalid="ignore"):
        cr = (mx - mn).astype(F32)
        s = cr / mx.astype(F32)
        rc, gc, bc = ((mx - c).astype(F32) / cr for c in (r, g, b))
        h = np.where(r == mx, bc - gc, np.where(g == mx, ((2.0 + rc.astype(F64)) - bc.astype(F64)).astype(F32),
                                                  ((4.0 + gc.astype(F64)) - rc.astype(F64)).astype(F32)))
        h = np.fmod(h.astype(F64) / 6.0 + 1.0, 1.0).astype(F32)
        H = np.clip((h.astype(F64) * 255.0).astype(np.int64), 0, 255)
        S = np.clip((s.astype(F64) * 255.0).astype(np.int64), 0, 255)
    return np.where(grey, 0, H), np.where(grey, 0, S), mx


def hsv2rgb(H, S, V):
    """Pillow's hsv2rgb (Convert.c) of int arrays -> (..., 3) uint8."""
    x = H.astype(F32).astype(F64) * 6.0 / 255.0
    i = np.floor(x).astype(np.int64)
    f = (x - i.astype(F32).astype(F64)).astype(F32)
    fs = (S.astype(F32).astype(F64) / 255.0).astype(F32)
    v = V.astype(F32).astype(F64)
    p = np.clip(_round(v * (1.0 - fs.astype(F64))), 0, 255)
    q = np.clip(_round(v * (1.0 - (fs * f).astype(F64))), 0, 255)
    t = np.clip(_round(v * (1.0 - fs.astype(F64) * (1.0 - f.astype(F64)))), 0, 255)
    k = i % 6
    sel = lambda *c: np.select([k == j for j in range(6)], c)
    out = np.stack([sel(V, q, p, p, t, V), sel(t, V, V, q, p, p), sel(p, p, t, V, V, q)], axis=-1)
    grey = (S == 0)[..., None]
    return np.where(grey, np.stack([V, V, V], axis=-1), out).astype(np.uint8)


def hue_shift(h):
    """The byte torchvision adds to H: np.array(h * 255).astype(np.uint8), i.e. truncated to int32, then wrapped."""
    return int(np.int32(h * 255.0).astype(np.uint8))


def _fields(col):
    return list(col.order), int(col.on), int(col.gray), list(col.factor)


def color_ref(px, col):
    """The (h, w, 3|4) uint8 array px after colour entry col (an xpngb_color, as color_params returns)."""
    order, on, gray, fac = _fields(col)
    out = px.copy()
    for k in order:
        if not (on >> k) & 1:
            continue
        rgb = out[..., :3]
        if k == 3:
            H, S, V = rgb2hsv(rgb)
            out[..., :3] = hsv2rgb((H + hue_shift(fac[3])) & 255, S, V)
            if out.shape[2] == 4:
                out[..., 3] = 255                     # adjust_hue goes through HSV, which has no alpha
            continue
        if k == 0:
            d = 0
        elif k == 1:
            L = luma(rgb)
            d = int(int(L.sum()) / L.size + 0.5)      # ImageStat: the float quotient of exact integer sums
        else:
            d = luma(rgb)[..., None]
        out[..., :3] = blend(d, rgb, fac[k])
    if gray:
        out[..., :3] = luma(out[..., :3])[..., None]
    return out


def col(order=(0, 1, 2, 3), b=None, c=None, s=None, h=None, gray=False):
    return color_params(list(order), b, c, s, h, gray)


# ---------------------------------------------------------------------------------------------------- oracle against PIL (CPU)

def _pil(px):
    return Image.fromarray(px, "RGBA" if px.shape[2] == 4 else "RGB")


def _quantised(rng, h, w, c):
    px = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
    if rng.random() < 0.3:   # few levels: maxima, minima and grey pixels tie
        px = (px // 85 * 85).astype(np.uint8)
    return px


def _boundary_factors(v):
    """Doubles just either side of the midpoint between float32 v and the next float32: Pillow narrows them to different
    floats."""
    lo, hi = float(F32(v)), float(np.nextafter(F32(v), F32(np.inf)))
    mid = (lo + hi) / 2
    return [np.nextafter(mid, -np.inf), np.nextafter(mid, np.inf)]


FACTORS = [0.0, 1.0, 2.5, 0.6, 1.4, 7.0] + _boundary_factors(0.7) + _boundary_factors(1.3)
HUES = [0.5, -0.5, 0.0, 0.5 / 255, -0.9 / 255, 0.1, -0.1, -0.3, 0.37, 1.0 / 255, -1.0 / 255]


@pytest.mark.parametrize("mode", ("RGB", "RGBA"))
def test_each_step_matches_torchvision(mode):
    """color_ref of each step alone against torchvision's PIL functional ops, seeded, sizes 1..69."""
    import torchvision.transforms.functional as F
    rng = np.random.default_rng(7 if mode == "RGB" else 8)
    c = 4 if mode == "RGBA" else 3
    fns = {0: F.adjust_brightness, 1: F.adjust_contrast, 2: F.adjust_saturation, 3: F.adjust_hue}
    cases = 0
    for k in range(4):
        vals = HUES if k == 3 else FACTORS + list(rng.uniform(0, 2, 6))
        for v in vals:
            for _ in range(6):
                h, w = int(rng.integers(1, 70)), int(rng.integers(1, 70))
                px = _quantised(rng, h, w, c)
                want = np.asarray(fns[k](_pil(px), float(v)))
                kw = {"bcsh"[k]: float(v)}
                got = color_ref(px, col(**kw))
                assert np.array_equal(got, want), (k, v, h, w)
                cases += 1
    for _ in range(20):   # grayscale of RGB
        px = _quantised(rng, int(rng.integers(1, 70)), int(rng.integers(1, 70)), 3)
        assert np.array_equal(color_ref(px, col(gray=True)), np.asarray(F.rgb_to_grayscale(_pil(px), 3)))
    assert cases > 300


def test_float32_narrowing_matters():
    """The boundary factors of FACTORS narrow to different floats, and the hue shifts truncate, then wrap."""
    a, b = _boundary_factors(1.3)
    assert F32(a) != F32(b)
    assert [hue_shift(h) for h in (0.5, -0.5, 0.5 / 255, -0.9 / 255, -0.3)] == [127, 129, 0, 0, 180]


def _all_colours():
    v = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], axis=-1).astype(np.uint8).reshape(4096, 4096, 3)


def test_rgb2hsv_exhaustive():
    """rgb2hsv against Image.convert("HSV") on all 2^24 RGB triples."""
    px = _all_colours()
    want = np.asarray(Image.fromarray(px, "RGB").convert("HSV"))
    for r0 in range(0, 4096, 1024):
        H, S, V = rgb2hsv(px[r0: r0 + 1024])
        got = np.stack([H, S, V], axis=-1).astype(np.uint8)
        assert np.array_equal(got, want[r0: r0 + 1024]), r0


def test_hsv2rgb_exhaustive():
    """hsv2rgb against Image.convert("RGB") of an HSV image holding all 2^24 HSV triples."""
    hsv = _all_colours()
    want = np.asarray(Image.frombytes("HSV", (4096, 4096), hsv.tobytes()).convert("RGB"))
    for r0 in range(0, 4096, 1024):
        part = hsv[r0: r0 + 1024].astype(np.int64)
        assert np.array_equal(hsv2rgb(part[..., 0], part[..., 1], part[..., 2]), want[r0: r0 + 1024]), r0


def replay_jitter(cj, rg_p=0.2, apply_p=0.8):
    """Draws what RandomApply([cj], apply_p) followed by RandomGrayscale(rg_p) draws, in the same order, and returns the
    colour entry (None: neither applies)."""
    import torch
    applied = not (apply_p < torch.rand(1))
    params = cj.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue) if applied else None
    gray = bool(torch.rand(1) < rg_p)
    if params is None and not gray:
        return None
    if params is None:
        return color_params([0, 1, 2, 3], None, None, None, None, gray)
    return color_params(*params, gray=gray)


def test_color_jitter_replay_matches_torchvision():
    """RandomApply([ColorJitter(0.4, 0.4, 0.2, 0.1)], 0.8) + RandomGrayscale(0.2) under a fixed seed equals color_ref fed by
    color_params of the replayed draws, for BYOL's and SimCLR's factors."""
    import torch
    import torchvision.transforms as T
    rng = np.random.default_rng(5)
    imgs = [_quantised(rng, int(rng.integers(1, 50)), int(rng.integers(1, 50)), 3) for _ in range(60)]
    for factors in ((0.4, 0.4, 0.2, 0.1), (0.8, 0.8, 0.8, 0.2)):
        cj = T.ColorJitter(*factors)
        tf = T.Compose([T.RandomApply([cj], p=0.8), T.RandomGrayscale(p=0.2)])
        torch.manual_seed(11)
        want = [np.asarray(tf(_pil(px))) for px in imgs]
        torch.manual_seed(11)
        cols = [replay_jitter(cj) for _ in imgs]
        for px, c, w in zip(imgs, cols, want):
            assert np.array_equal(px if c is None else color_ref(px, c), w)
        assert sum(c is not None and c.gray for c in cols) > 3 and sum(c is not None and c.on == 15 for c in cols) > 20


def test_contrast_mean_half_way():
    """Contrast on images whose mean luma is exactly k + 0.5 (rounds up) and one step below it (rounds down)."""
    import torchvision.transforms.functional as F
    for k in (0, 17, 127, 200):
        for extra in (1, 0):   # luma sum k * N + N / 2 (+ 0 or - 1 over N = 64)
            L = np.full(64, k, np.int64)
            L[:32] += 1
            if not extra:
                L[0] -= 1
            px = np.repeat(L.astype(np.uint8)[:, None], 3, axis=1).reshape(8, 8, 3)
            assert int(luma(px).sum()) == 64 * k + 32 - (1 - extra)
            for f in (0.5, 1.7, 0.0):
                want = np.asarray(F.adjust_contrast(_pil(px), f))
                assert np.array_equal(color_ref(px, col(c=f)), want), (k, extra, f)
            assert np.array_equal(np.unique(color_ref(px, col(c=0.0))), [k + extra])


@pytest.mark.parametrize("op", ALL_OPS)
def test_steps_commute_with_the_op(op):
    """Every step is per pixel and the contrast mean ignores pixel order: colour before and after each op agree."""
    rng = np.random.default_rng(ALL_OPS.index(op))
    for c in (3, 4):
        px = _quantised(rng, 37, 53, c)
        for _ in range(6):
            cc = col(rng.permutation(4), *rng.uniform(0, 2, 3), float(rng.uniform(-0.5, 0.5)), gray=(c == 3 and rng.random() < 0.5))
            assert np.array_equal(color_ref(po.orient(op, px), cc), po.orient(op, color_ref(px, cc)))


def test_color_params_fields():
    import torch
    c = color_params(torch.tensor([3, 0, 2, 1]), 1.2, None, 0.7, -0.05, gray=True)
    assert list(c.order) == [3, 0, 2, 1] and c.on == 0b1101 and c.gray == 1 and list(c.factor) == [1.2, 1.0, 0.7, -0.05]
    arr = color_array([None, c], 2)
    assert list(arr[0].order) == [0, 1, 2, 3] and arr[0].on == 0 and arr[0].gray == 0 and arr[1].on == 0b1101
    assert C.sizeof(_Color) == 48


# ---------------------------------------------------------------------------------------------------- colour decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def random_col(rng, gray_ok=True, order=None):
    return col(rng.permutation(4) if order is None else order, *rng.uniform(0, 2, 3), float(rng.uniform(-0.5, 0.5)),
               gray=gray_ok and rng.random() < 0.5)


def entry_ref(full, c, rect=None, size=None, filt=2, win=None, op=None):
    px = full if rect is None else window(full, rect)
    if size is not None:
        px = window(resize_pil(px, size[0], size[1], filt), win)
    px = po.orient(op or "tl", px)
    return px if c is None else color_ref(px, c)


def check_u8(cd, files, fulls, cols, boxes=None, szs=None, ops=None, filters=None, wins=None):
    if szs is not None:
        got = cd.decode_resized(files, szs, boxes, ops, filters, wins, colors=cols)
    else:   # no resize: through decode_color_raw
        n = len(files)
        nb = [(boxes[i][2] * boxes[i][3] if boxes else fulls[i].shape[0] * fulls[i].shape[1]) * fulls[i].shape[2] for i in range(n)]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.zeros(poff + 16, np.uint8)
        cd.decode_color_raw(None, descs, None, None if ops is None else op_codes(ops), None if boxes is None else rects(boxes), None, None,
                            color_array(cols, n), n, fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
        got = []
        for i in range(n):
            h, w = (boxes[i][3], boxes[i][2]) if boxes else fulls[i].shape[:2]
            if ops is not None and ops[i] in ("r90", "r270"):
                h, w = w, h
            got.append(out[descs[i].offset: descs[i].offset + nb[i]].reshape(h, w, fulls[i].shape[2]))
    for i, g in enumerate(got):
        want = entry_ref(fulls[i], cols[i], None if boxes is None else boxes[i], None if szs is None else szs[i],
                         2 if filters is None else filters[i], None if wins is None else wins[i], None if ops is None else ops[i])
        assert g.shape == want.shape and np.array_equal(g, want), (i, cols[i] and _fields(cols[i]))


ORDERS = [list(p) for p in __import__("itertools").permutations(range(4))]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_orders_steps_and_geometry(codec, level):
    """All 24 orders with every step on, gray on and off; each step alone; crops, the seven ops, resizes with the five filters
    and windows; RGB and RGBA (whose entries get no gray: their uint8 output keeps alpha)."""
    rng = np.random.default_rng(40 + level)
    imgs = [synth.rgb(300, 420, level), synth.rgba(260, 310, level + 9)]
    files = [po.encode(level, im) for im in imgs]
    fulls = [po.decode(f) for f in files]
    assert [x.shape[2] for x in fulls] == [3, 4]
    for k, (f, full) in enumerate(zip(files, fulls)):
        h, w = full.shape[:2]
        a = full.shape[2] == 4
        cols = [col(o, *rng.uniform(0, 2, 3), float(rng.uniform(-0.5, 0.5)), gray=not a and g) for o in ORDERS for g in (False, True)]
        cols += [col(b=0.0), col(c=0.0), col(s=0.0), col(b=1.6), col(c=1.9), col(s=2.0), col(h=0.5), col(h=-0.5), col(h=0.2),
                 None, col(gray=not a)]
        n = len(cols)
        boxes = [(int(x), int(y), int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1)))
                 for x, y in zip(rng.integers(0, w, n), rng.integers(0, h, n))]
        ops = [ALL_OPS[j % 7] for j in range(n)]
        check_u8(codec, [f] * n, [full] * n, cols, boxes, None, ops)          # crops and ops, no resize
        check_u8(codec, [f] * 4, [full] * 4, cols[:4])                         # whole images
        szs = [(int(rng.integers(1, 300)), int(rng.integers(1, 300))) for _ in range(n)]
        wins = []
        for z in szs:
            x, y = int(rng.integers(z[0])), int(rng.integers(z[1]))
            wins.append((x, y, int(rng.integers(1, z[0] - x + 1)), int(rng.integers(1, z[1] - y + 1))))
        filters = [FILTERS[j % 5] for j in range(n)]
        check_u8(codec, [f] * n, [full] * n, cols, boxes, szs, ops, filters, wins)


TENSOR_FORMATS = [(dt, lay, da) for dt in ("float32", "float16", "bfloat16", "uint8") for lay in ("chw", "hwc") for da in (False, True)]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_tensor_formats(codec, level):
    """float32, float16, bfloat16 and uint8 tensors in CHW and HWC, alpha kept and dropped, resized and not: every element
    is to_tensor_ref of color_ref's pixels."""
    import torch
    rng = np.random.default_rng(70 + level)
    for im in (synth.rgb(200, 260, level + 30), synth.rgba(180, 240, level + 31)):
        f = po.encode(level, im)
        full = po.decode(f)
        a = full.shape[2] == 4
        for dt, lay, da in TENSOR_FORMATS:
            n = 6
            cols = [random_col(rng, gray_ok=da or not a) for _ in range(n - 1)] + [None]
            ops = [ALL_OPS[int(rng.integers(7))] for _ in range(n)]
            boxes = [(10, 5, 64, 64)] * n
            for szs in (None, [(32, 32)] * n):
                got = codec.decode_tensor([f] * n, szs, boxes, ["tl"] * n, getattr(torch, dt), lay, mean=IMAGENET["mean"],
                                          std=IMAGENET["std"], drop_alpha=da, filters=None if szs is None else [FILTERS[j % 5] for j in range(n)],
                                          colors=cols)
                for i in range(n):
                    want = to_tensor_ref(entry_ref(full, cols[i], boxes[i], None if szs is None else szs[i], FILTERS[i % 5] if szs else 2),
                                         dt, lay, "div", IMAGENET["mean"], IMAGENET["std"], da)
                    assert np.array_equal(bits(got[i]), want), (dt, lay, da, szs is None, i)
            # ragged, with ops and windows
            szs = [(int(rng.integers(8, 90)), int(rng.integers(8, 90))) for _ in range(n)]
            wins = [(1, 2, z[0] - 3, z[1] - 2) for z in szs]
            fmt = tensor_format(dt, lay, "mul", IMAGENET["mean"], IMAGENET["std"], da)
            eb = {"uint8": 1, "float32": 4, "float16": 2, "bfloat16": 2}[dt]
            C_ = 3 if da else full.shape[2]
            nb = [ww * wh * C_ * eb for (_, _, ww, wh) in wins]
            descs, foffs, fsizes, fb, poff = pack([f] * n, nb)
            fa = np.frombuffer(fb, np.uint8)
            out = np.zeros(poff + 16, np.uint8)
            codec.decode_color_raw(fmt, descs, filter_codes("bicubic", n), op_codes(ops), rects(boxes), size_arr(szs), rects(wins),
                                   color_array(cols, n), n, fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
            for i in range(n):
                want = to_tensor_ref(entry_ref(full, cols[i], boxes[i], szs[i], 3, wins[i], ops[i]), dt, lay, "mul",
                                     IMAGENET["mean"], IMAGENET["std"], da)
                got = out[descs[i].offset: descs[i].offset + nb[i]].view(want.dtype).reshape(want.shape)
                assert np.array_equal(got, want), (dt, lay, da, "ragged", i)


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_torchvision_byol_pipeline(codec, level):
    """One seeded batch bit-identical to Compose([RandomResizedCrop(224), RandomHorizontalFlip(), RandomApply([ColorJitter(0.4,
    0.4, 0.2, 0.1)], 0.8), RandomGrayscale(0.2), ToTensor(), Normalize(ImageNet)]) on PIL images, the RNG replayed."""
    import torch
    import torchvision.transforms as T
    imgs = [synth.rgb(h, w, 900 + k) for k, (w, h) in enumerate([(500, 375), (333, 500), (640, 427), (300, 300)] * 4)]
    files = [po.encode(level, im) for im in imgs]
    cj = T.ColorJitter(0.4, 0.4, 0.2, 0.1)
    rrc = T.RandomResizedCrop(224)
    tf = T.Compose([rrc, T.RandomHorizontalFlip(), T.RandomApply([cj], p=0.8), T.RandomGrayscale(p=0.2), T.ToTensor(),
                    T.Normalize(*IMAGENET.values())])
    torch.manual_seed(2024 + level)
    want = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    torch.manual_seed(2024 + level)
    boxes, ops, cols = [], [], []
    for im in imgs:
        i, j, h, w = T.RandomResizedCrop.get_params(Image.fromarray(im), rrc.scale, rrc.ratio)
        boxes.append((j, i, w, h))
        ops.append("mh" if torch.rand(1) < 0.5 else "tl")
        cols.append(replay_jitter(cj))
    got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, torch.float32, mean=IMAGENET["mean"], std=IMAGENET["std"],
                              colors=cols).cpu()
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


@gpu
def test_every_colour_hue_shifts(codec):
    """A 4096 x 4096 image holding every RGB colour, hue-shifted by every reachable kind of shift, on every pixel."""
    px = _all_colours()
    f = codec.encode(1, [px])[0]
    for k in (1, 26, 127, 129, 230, 255):   # 128 is unreachable: |h| <= 0.5 gives shifts in [-127, 127]
        h = (k + 0.5) / 255 if k < 128 else (k - 256 - 0.5) / 255
        c = col(h=h)
        assert hue_shift(h) == k
        got = codec.decode_resized([f], [(4096, 4096)], colors=[c])[0]
        want = np.empty_like(px)
        for r0 in range(0, 4096, 1024):
            want[r0: r0 + 1024] = color_ref(px[r0: r0 + 1024], c)
        assert np.array_equal(got, want), k


@gpu
def test_contrast_8k_sum_exceeds_32_bits(codec):
    """Contrast of a whole 8192 x 8192 entry, whose luma sum exceeds 2^32, after brightness moved it."""
    import torch
    rng = np.random.default_rng(8)
    tile = rng.integers(150, 256, (64, 64, 3), dtype=np.uint8)
    px = np.tile(tile, (128, 128, 1))
    f = codec.encode(1, [px])[0]
    c = col([0, 1, 2, 3], b=0.93, c=0.41)
    bright = color_ref(px[:64, :64], col(b=0.93))
    assert int(luma(bright).sum()) * 128 * 128 > 1 << 32
    got = codec.decode_tensor([f], None, None, None, torch.uint8, "hwc", colors=[c]).cpu().numpy()[0]
    # the chain on the tile equals the chain on the image: the same mean
    want_tile = color_ref(px[:64, :64], c)
    assert np.array_equal(got, np.tile(want_tile, (128, 128, 1)))


@gpu
def test_pipelined_chunks_device_resident(monkeypatch):
    """Sintel-like frames cut into at least 3 chunks on 2 lanes, files and output in device memory, uint8 and float32."""
    import torch
    frames = synth.sintel_batch(range(2000, 2008))
    for k, v in (("XPNGB_LAT_MAX_BLOCKS", "0"), ("XPNGB_PIPE_MIN_MPIX", "1"), ("XPNGB_PIPE_LANES", "2"), ("XPNGB_CHUNK_MPIX", "3")):
        monkeypatch.setenv(k, v)
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(99)
        n = len(frames)
        boxes = [(int(rng.integers(0, 900)), int(rng.integers(0, 500)), 1000, 500) for _ in range(n)]
        szs = [(224, 224) if k % 2 else None for k in range(n)]
        cols = [random_col(rng) if k != 3 else None for k in range(n)]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for fmt, eb in ((None, 1), (tensor_format("float32", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True), 4)):
                nb = [(224 * 224 if z else b[2] * b[3]) * 3 * eb for z, b in zip(szs, boxes)]
                descs, foffs, fsizes, fb, poff = pack(files, nb)
                dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
                dout = torch.zeros(poff, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                zs = [z or (b[2], b[3]) for z, b in zip(szs, boxes)]   # an entry whose size equals its crop is the crop
                cd.profile(True)
                cd.decode_color_raw(fmt, descs, None, None, rects(boxes), size_arr(zs), None, color_array(cols, n), n, dfiles.data_ptr(),
                                    len(fb), 1, foffs, fsizes, dout.data_ptr(), poff, 1)
                rep = cd.profile_report()
                cd.profile(False)
                assert rep["k_color"][1] >= 3 and "k_color_mean" in rep, rep
                out = dout.cpu().numpy()
                for i in range(n):
                    px = entry_ref(frames[i], cols[i], boxes[i], szs[i])
                    want = px if fmt is None else to_tensor_ref(px, "float32", "chw", "div", IMAGENET["mean"], IMAGENET["std"], True)
                    got = out[descs[i].offset: descs[i].offset + nb[i]]
                    assert np.array_equal(got, want.reshape(-1).view(np.uint8)), (lv, fmt is None, i)
    finally:
        cd.close()


@gpu
def test_null_and_empty_colours_are_the_existing_calls(codec):
    """colors == NULL and all-empty programs give the bytes of decode_resampled, decode_tensor and decode_oriented."""
    import torch
    imgs = [synth.rgb(300, 400, 1), synth.rgba(200, 260, 2), synth.rgb(123, 77, 3)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)]
    boxes = [(5, 6, 200, 150), (0, 0, 260, 200), (1, 1, 70, 100)]
    ops = ["r90", "mh", "tl"]
    empty = [None, col(), col([3, 2, 1, 0])]
    base = codec.decode_resized(files, [(64, 48)] * 3, boxes, ops, "bicubic", [(2, 2, 50, 40)] * 3)
    for cols in (None, empty):
        got = codec.decode_resized(files, [(64, 48)] * 3, boxes, ops, "bicubic", [(2, 2, 50, 40)] * 3, colors=cols or [None] * 3)
        assert all(np.array_equal(a, b) for a, b in zip(got, base))
    t0 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, torch.bfloat16, "hwc", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True)
    t1 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, torch.bfloat16, "hwc", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True,
                             colors=empty)
    assert torch.equal(t0.view(torch.int16), t1.view(torch.int16))
    want = codec.decode_region(files, boxes, ops)
    for cols in (None, empty):
        nb = [b[2] * b[3] * im.shape[2] for b, im in zip(boxes, imgs)]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.zeros(poff + 16, np.uint8)
        codec.decode_color_raw(None, descs, None, op_codes(ops), rects(boxes), None, None, color_array(cols, 3), 3, fa.ctypes.data,
                               len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
        for i, w in enumerate(want):
            assert out[descs[i].offset: descs[i].offset + w.size].tobytes() == w.tobytes()


@gpu
def test_color_failures(codec):
    """Each refused input fails naming the entry, before anything is written."""
    px, pa = synth.rgb(100, 120, 5), synth.noise(90, 80, 6, channels=4)   # random alpha: the file keeps it
    f, fa_ = po.encode(1, px), po.encode(2, pa)
    assert po.decode(fa_).shape[2] == 4

    def call(c1, files=None, fmt=None, szs=None, filters=None, wins=None):
        files = files or [f, f]
        nb = [100 * 120 * 4 * 4] * 2
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, 0xA5, np.uint8)
        cols = color_array([col(b=1.2), c1], 2)
        err = None
        try:
            codec.decode_color_raw(fmt, descs, filters, None, None, szs, wins, cols, 2, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                   out.ctypes.data, poff, 0)
        except RuntimeError as e:
            err = str(e)
        return err, out

    bad = []
    for order in ([0, 1, 2, 2], [0, 1, 2, 4], [3, 3, 3, 3]):
        bad.append((col(order, b=1.0), "order"))
    c = col(b=1.0); c.on = 0b10001; bad.append((c, "above 3"))
    c = col(); c.gray = 2; bad.append((c, "gray"))
    for v in (-0.1, math.inf, math.nan, 1e300):
        for k in "bcs":
            bad.append((col(**{k: v}), "factor"))
    for v in (0.5000001, -0.51, math.nan, math.inf):
        bad.append((col(h=v), "hue"))
    for c1, word in bad:
        err, out = call(c1)
        assert err is not None and "entry 1" in err and word in err and (out == 0xA5).all(), (_fields(c1), err)
    for fmt in (None, tensor_format("float32")):   # gray on an RGBA entry whose output keeps alpha
        err, out = call(col(gray=True), [f, fa_], fmt)
        assert err is not None and "entry 1" in err and "alpha" in err and (out == 0xA5).all(), err
    assert call(col(gray=True), [f, fa_], tensor_format("float32", drop_alpha=True))[0] is None
    err, out = call(col(b=0.5), filters=filter_codes("bicubic", 2))      # filters without sizes
    assert err is not None and "sizes" in err and (out == 0xA5).all()
    err, out = call(col(b=0.5), wins=rects([(0, 0, 5, 5)] * 2))
    assert err is not None and "sizes" in err and (out == 0xA5).all()
    assert call(col(b=0.5))[0] is None
