"""Blurred and solarized decode (xpngb_decode_blur / Codec.decode_resized and decode_tensor with blurs): Pillow's
ImageFilter.GaussianBlur and ImageOps.solarize applied to each entry after its colour step, byte-identical to Pillow.  Entry i
is tensor(solarize_i(blur_i(gray_i(jitter_i(orient(op_i, window_i(resize_f(crop_i)))))))).

blur_pil() restates Pillow's BoxBlur.c in numpy (float box radius, three uint32 box passes per axis, x before y); the CPU tests
pin it, box_ref() and solarize_ref() to the installed Pillow.  On the GPU every output is compared with Pillow itself applied
to po.decode's pixels."""
import math
import random

import numpy as np
import pytest
from PIL import Image, ImageFilter, ImageOps

from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import (_Blur, blur_array, blur_box, blur_params, color_array, filter_codes, op_codes, rects,
                             sizes as size_arr, tensor_format)
from test_color_decode import col, entry_ref, random_col, replay_jitter
from test_resampled_decode import FILTERS, pack
from test_tensor_decode import IMAGENET, bits, to_tensor_ref

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
F32 = np.float32
RADIUS_MAX = 8388608.0   # XPNGB_BLUR_RADIUS_MAX


# ---------------------------------------------------------------------------------------------------- the oracle

def box_ref(radius):
    """(ri, ww, fw) of one axis, as Pillow's _gaussian_blur_radius + ImagingHorizontalBoxBlur compute them in float, for an
    array of radii.  fw is the uint32 Pillow stores (it wraps when (2 ri + 1) * ww > 2^24)."""
    r = np.asarray(radius, dtype=np.float64).astype(F32)
    s2 = (r * r / F32(3)).astype(F32)
    L = np.sqrt((s2 * F32(12) + F32(1)).astype(F32).astype(np.float64)).astype(F32)
    l = np.floor(((L - F32(1)) / F32(2)).astype(F32))
    a = ((F32(2) * l + F32(1)) * (l * (l + F32(1)) - F32(3) * s2)).astype(F32)
    a = (a / (F32(6) * (s2 - (l + F32(1)) * (l + F32(1))))).astype(F32)
    fr = (l + a).astype(F32)
    ri = fr.astype(np.int64)
    ww = (F32(16777216) / (fr * F32(2) + F32(1))).astype(F32).astype(np.int64)
    fw = (((1 << 24) - (2 * ri + 1) * ww) % (1 << 32)) // 2
    return ri, ww, fw


def _box_pass(px, ri, ww, fw):
    """One box pass along axis 1 of an (h, w, c) uint8 array: edges clamped, Pillow's uint32 arithmetic (checked not to wrap)."""
    w = px.shape[1]
    idx = np.clip(np.arange(-ri - 1, w + ri + 1), 0, w - 1)
    p = px[:, idx, :].astype(np.uint64)                       # padded by ri + 1 on each side
    cs = np.concatenate([np.zeros_like(p[:, :1]), np.cumsum(p, axis=1)], axis=1)
    x = np.arange(w)
    acc = cs[:, x + 2 * ri + 2] - cs[:, x + 1]                # p[x - ri .. x + ri]
    bulk = acc * ww + (p[:, x] + p[:, x + 2 * ri + 2]) * fw
    assert (bulk + (1 << 23) < 1 << 32).all()
    return ((bulk + (1 << 23)) >> 24).astype(np.uint8)


def blur_pil(px, rx, ry, order="xy"):
    """ImageFilter.GaussianBlur((rx, ry)) of the (h, w, c) uint8 array px: three passes along x, then three along y (order
    "yx": y first).  An axis whose float radius is 0 is skipped."""
    out = px
    for ax in order:
        r = rx if ax == "x" else ry
        if F32(r) == 0:
            continue
        ri, ww, fw = (int(v) for v in box_ref(r))
        for _ in range(3):
            out = _box_pass(out, ri, ww, fw) if ax == "x" else _box_pass(out.transpose(1, 0, 2), ri, ww, fw).transpose(1, 0, 2)
    return np.ascontiguousarray(out)


def solarize_t(threshold):
    """The library's solarize rule: bytes below clamp(ceil(threshold), 0, 256) are kept."""
    c = math.ceil(threshold) if math.isfinite(threshold) else threshold
    return 0 if c <= 0 else 256 if c >= 256 else int(c)


def solarize_ref(px, threshold):
    t = solarize_t(threshold)
    return np.where(px < t, px, 255 - px).astype(np.uint8)


def _pil(px):
    return Image.fromarray(px, "RGBA" if px.shape[2] == 4 else "RGB")


def pil_blur(px, b):
    """px after the blur entry b (an xpngb_blur) as Pillow computes it; solarize of RGBA (alpha dropped later) by solarize_ref."""
    if b is None:
        return px
    out = px
    if tuple(b.radius) != (0.0, 0.0):
        out = np.asarray(_pil(px).filter(ImageFilter.GaussianBlur(tuple(b.radius))))
    if b.solarize:
        out = np.asarray(ImageOps.solarize(_pil(out), b.threshold)) if out.shape[2] == 3 else solarize_ref(out, b.threshold)
    return out


# ---------------------------------------------------------------------------------------------------- oracle against PIL (CPU)

def _ri_steps(kmax):
    """For k = 1 .. kmax, the smallest float32 radius whose box radius is k (bisection over float32 bit patterns)."""
    out = []
    for k in range(1, kmax + 1):
        lo, hi = int(F32(0.01).view(np.int32)), int(F32(4 * k + 4).view(np.int32))
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if box_ref(np.int32(mid).view(F32))[0] >= k:
                hi = mid
            else:
                lo = mid
        out.append((float(np.int32(lo).view(F32)), float(np.int32(hi).view(F32))))
    return out


RI_STEPS = _ri_steps(12)


def test_ri_steps_are_where_ri_changes():
    for k, (below, at) in enumerate(RI_STEPS, 1):
        assert box_ref(below)[0] == k - 1 and box_ref(at)[0] == k, (k, below, at)


def test_blur_pil_matches_pillow():
    """blur_pil equals ImageFilter.GaussianBlur on RGB and RGBA: sizes from 1 x 1, 1 x N and N x 1 up to 69 x 69, radii in
    [0.1, 2], above the image side and 1e4, per-axis radii with one axis 0, and the float32 radii either side of each
    point where ri changes."""
    rng = np.random.default_rng(0)
    radii = [(float(rng.uniform(0.1, 2.0)),) * 2 for _ in range(200)]
    radii += [(float(rng.uniform(70, 200)),) * 2 for _ in range(30)] + [(1e4, 1e4), (1e4, 0.7), (0.0, 1e4)]
    radii += [(float(rng.uniform(0.1, 9)), 0.0) for _ in range(30)] + [(0.0, float(rng.uniform(0.1, 9))) for _ in range(30)]
    radii += [(float(rng.uniform(0.1, 9)), float(rng.uniform(0.1, 9))) for _ in range(60)]
    for below, at in RI_STEPS:
        radii += [(below, below), (at, at), (below, at), (at, 0.0)]
    sizes = [(1, 1), (1, 37), (37, 1), (1, 2), (2, 1)]
    cases = 0
    for k, (rx, ry) in enumerate(radii):
        c = 4 if k % 2 else 3
        h, w = sizes[k] if k < len(sizes) else (int(rng.integers(1, 70)), int(rng.integers(1, 70)))
        px = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
        if k % 4 == 0:   # blocky: long runs of equal bytes
            px = np.repeat(np.repeat(px[::8, ::8], 8, 0), 8, 1)[:h, :w]
            px = np.ascontiguousarray(np.pad(px, ((0, h - px.shape[0]), (0, w - px.shape[1]), (0, 0)), mode="edge"))
        want = np.asarray(_pil(px).filter(ImageFilter.GaussianBlur((rx, ry))))
        assert np.array_equal(blur_pil(px, rx, ry), want), (k, rx, ry, h, w, c)
        cases += 1
    assert cases >= 400


def test_blur_box_matches_pillows_arithmetic():
    """xpngb_blur_box equals box_ref on 120,000 radii (log-uniform over 1e-3 .. 2^23, plus the ri steps and the bound)."""
    rng = np.random.default_rng(1)
    radii = list(np.exp(rng.uniform(math.log(1e-3), math.log(RADIUS_MAX), 120000)))
    radii += [r for pair in RI_STEPS for r in pair] + [0.1, 2.0, 1e4, 1e6, RADIUS_MAX, float(np.nextafter(F32(RADIUS_MAX), F32(0)))]
    ri, ww, fw = box_ref(radii)
    for k, r in enumerate(radii):
        assert blur_box(r) == (ri[k], ww[k], fw[k]), r


def test_radius_bound():
    """The refusal bound is where Pillow's uint32 box sums could first wrap: up to float radius 2^23 (2 ri + 1) * ww <= 2^24,
    so acc * ww + far * fw + 2^23 stays below 2^32; at 8388609, ri = 2^23, ww = 1 and fw wraps."""
    bits_ = np.arange(int(F32(RADIUS_MAX).view(np.int32)) - 2_000_000, int(F32(RADIUS_MAX).view(np.int32)) + 1, dtype=np.int32)
    for r in (bits_.view(F32), np.exp(np.random.default_rng(2).uniform(math.log(1e-6), math.log(RADIUS_MAX), 2_000_000))):
        ri, ww, fw = box_ref(r)
        assert ((2 * ri + 1) * ww <= 1 << 24).all() and (255 * ((2 * ri + 1) * ww + 2 * fw) + (1 << 23) < 1 << 32).all()
        assert (255 * (2 * ri + 1) < 1 << 32).all()
    ri, ww, fw = (int(v) for v in box_ref(8388609.0))
    assert (ri, ww) == (1 << 23, 1) and (2 * ri + 1) * ww > 1 << 24 and fw > 1 << 30
    assert blur_box(RADIUS_MAX) is not None and blur_box(8388608.4) is not None    # 8388608.4 narrows to 2^23
    for r in (8388609.0, 8388608.6, 1e30, math.inf, math.nan, -0.5, -1e-30):
        assert blur_box(r) is None, r


@pytest.mark.parametrize("op", ALL_OPS)
def test_blur_and_the_op(op):
    """blur(op(x), rx, ry) == op(blur of x with the axes' passes in x's own frame): mirrors commute, quarter turns need the
    y passes first with rx, then the x passes with ry."""
    rng = np.random.default_rng(ALL_OPS.index(op) + 10)
    for k in range(12):
        h, w = int(rng.integers(1, 60)), int(rng.integers(1, 60))
        rx, ry = float(rng.uniform(0.1, 6)), float(rng.uniform(0.1, 6)) if k % 3 else 0.0
        x = rng.integers(0, 256, (h, w, 3 + k % 2), dtype=np.uint8)
        lhs = blur_pil(np.ascontiguousarray(po.orient(op, x)), rx, ry)
        if op in ("r90", "r270"):
            rhs = po.orient(op, blur_pil(x, ry, rx, order="yx"))
        else:
            rhs = po.orient(op, blur_pil(x, rx, ry))
        assert np.array_equal(lhs, rhs), (op, k)


def test_pass_order_matters():
    """x passes then y passes differ from y then x: the swap of the quarter turns is needed."""
    rng = np.random.default_rng(3)
    xs = [rng.integers(0, 256, (40, 40, 3), dtype=np.uint8) for _ in range(20)]
    assert all(not np.array_equal(blur_pil(x, 1.3, 1.3), blur_pil(x, 1.3, 1.3, "yx")) for x in xs)


def test_solarize_matches_pillow():
    rng = np.random.default_rng(4)
    px = np.concatenate([np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, 2),
                         rng.integers(0, 256, (16, 16, 3), dtype=np.uint8)])
    for t in (-1, 0, 0.5, 127.5, 128, 255, 256, math.inf, -math.inf, 1e9, 254.0001):
        assert np.array_equal(solarize_ref(px, t), np.asarray(ImageOps.solarize(_pil(px), t))), t
    with pytest.raises(OSError):
        ImageOps.solarize(_pil(np.zeros((2, 2, 4), np.uint8)))


def test_blur_params_fields():
    b = blur_params(1.5, 128)
    assert list(b.radius) == [1.5, 1.5] and b.solarize == 1 and b.threshold == 128.0
    b = blur_params((0, 2.5))
    assert list(b.radius) == [0.0, 2.5] and b.solarize == 0
    arr = blur_array([None, b], 2)
    assert list(arr[0].radius) == [0.0, 0.0] and arr[0].solarize == 0 and list(arr[1].radius) == [0.0, 2.5]
    import ctypes as C
    assert C.sizeof(_Blur) == 32


# ---------------------------------------------------------------------------------------------------- blurred decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def random_blur(rng, solarize_ok=True):
    k = rng.random()
    radius = None if k < 0.15 else float(rng.uniform(0.1, 2.0)) if k < 0.7 else (float(rng.uniform(0, 5)), float(rng.uniform(0, 5)))
    thr = float(rng.choice([128, 0.5, 200.7, -3, 300])) if solarize_ok and rng.random() < 0.5 else None
    return blur_params(radius, thr)


def blur_entry_ref(full, c, b, rect=None, size=None, filt=2, win=None, op=None):
    return pil_blur(entry_ref(full, c, rect, size, filt, win, op), b)


def _out_hw(boxes, szs, wins, fulls, ops, i):
    if wins is not None:
        w, h = wins[i][2], wins[i][3]
    elif szs is not None:
        w, h = szs[i]
    elif boxes is not None:
        w, h = boxes[i][2], boxes[i][3]
    else:
        h, w = fulls[i].shape[:2]
    return (w, h) if ops is not None and ops[i] in ("r90", "r270") else (h, w)


def check_u8(cd, files, fulls, cols, blurs, boxes=None, szs=None, ops=None, filters=None, wins=None):
    """uint8 output through decode_blur_raw against Pillow's chain."""
    n = len(files)
    hw = [_out_hw(boxes, szs, wins, fulls, ops, i) for i in range(n)]
    nb = [h * w * fulls[i].shape[2] for i, (h, w) in enumerate(hw)]
    descs, foffs, fsizes, fb, poff = pack(files, nb)
    fa = np.frombuffer(fb, np.uint8)
    out = np.zeros(poff + 16, np.uint8)
    cd.decode_blur_raw(None, descs, None if filters is None else filter_codes(filters, n), None if ops is None else op_codes(ops),
                       None if boxes is None else rects(boxes), None if szs is None else size_arr(szs), None if wins is None else rects(wins),
                       None if cols is None else color_array(cols, n), blur_array(blurs, n), n, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                       out.ctypes.data, poff, 0)
    for i in range(n):
        got = out[descs[i].offset: descs[i].offset + nb[i]].reshape(hw[i][0], hw[i][1], fulls[i].shape[2])
        want = blur_entry_ref(fulls[i], None if cols is None else cols[i], blurs[i], None if boxes is None else boxes[i],
                              None if szs is None else szs[i], 2 if filters is None else filters[i], None if wins is None else wins[i],
                              None if ops is None else ops[i])
        assert np.array_equal(got, want), (i, blurs[i] and (list(blurs[i].radius), blurs[i].solarize, blurs[i].threshold))


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_blur_geometry(codec, level):
    """Seeded radii and thresholds, with and without colour: crops under all seven ops, whole images, resizes with the five
    filters and windows; RGB and RGBA (whose uint8 entries are not solarized: they keep alpha)."""
    rng = np.random.default_rng(140 + level)
    imgs = [synth.rgb(300, 420, level), synth.rgba(260, 310, level + 9)]
    files = [po.encode(level, im) for im in imgs]
    fulls = [po.decode(f) for f in files]
    assert [x.shape[2] for x in fulls] == [3, 4]
    for f, full in zip(files, fulls):
        h, w = full.shape[:2]
        a = full.shape[2] == 4
        n = 28
        blurs = [random_blur(rng, not a) for _ in range(n)]
        blurs[:7] = [blur_params(float(rng.uniform(0.1, 2.0)), None if a else 128) for _ in range(7)]   # every op blurred
        cols = [random_col(rng, gray_ok=not a) if k % 2 else None for k in range(n)]
        boxes = [(int(x), int(y), int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1)))
                 for x, y in zip(rng.integers(0, w, n), rng.integers(0, h, n))]
        ops = [ALL_OPS[j % 7] for j in range(n)]
        check_u8(codec, [f] * n, [full] * n, cols, blurs, boxes, None, ops)          # crops and ops, no resize
        check_u8(codec, [f] * n, [full] * n, None, blurs, boxes, None, ops)          # without colour
        check_u8(codec, [f] * 3, [full] * 3, cols[:3], blurs[:3])                    # whole images
        szs = [(int(rng.integers(1, 300)), int(rng.integers(1, 300))) for _ in range(n)]
        wins = []
        for z in szs:
            x, y = int(rng.integers(z[0])), int(rng.integers(z[1]))
            wins.append((x, y, int(rng.integers(1, z[0] - x + 1)), int(rng.integers(1, z[1] - y + 1))))
        filters = [FILTERS[j % 5] for j in range(n)]
        check_u8(codec, [f] * n, [full] * n, cols, blurs, boxes, szs, ops, filters, wins)


TENSOR_FORMATS = [(dt, lay, da) for dt in ("float32", "float16", "bfloat16", "uint8") for lay in ("chw", "hwc") for da in (False, True)]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_tensor_formats(codec, level):
    """Every tensor format, alpha kept and dropped, resized and not, each of the seven ops (quarter turns included): every
    element is to_tensor_ref of Pillow's blurred and solarized pixels."""
    import torch
    rng = np.random.default_rng(170 + level)
    for im in (synth.rgb(200, 260, level + 30), synth.rgba(180, 240, level + 31)):
        f = po.encode(level, im)
        full = po.decode(f)
        a = full.shape[2] == 4
        for dt, lay, da in TENSOR_FORMATS:
            n = 7
            sol = da or not a
            blurs = [random_blur(rng, sol) for _ in range(n - 1)] + [None]
            blurs[0] = blur_params((0.3, 4.1), 128 if sol else None)
            cols = [random_col(rng, gray_ok=sol) if k % 2 else None for k in range(n)]
            ops = ALL_OPS[:]
            boxes = [(10, 5, 64, 64)] * n
            for szs in (None, [(32, 32)] * n):
                got = codec.decode_tensor([f] * n, szs, boxes, ops, getattr(torch, dt), lay, mean=IMAGENET["mean"], std=IMAGENET["std"],
                                          drop_alpha=da, filters=None if szs is None else [FILTERS[j % 5] for j in range(n)],
                                          colors=cols, blurs=blurs)
                for i in range(n):
                    px = blur_entry_ref(full, cols[i], blurs[i], boxes[i], None if szs is None else szs[i], FILTERS[i % 5] if szs else 2,
                                        None, ops[i])
                    want = to_tensor_ref(px, dt, lay, "div", IMAGENET["mean"], IMAGENET["std"], da)
                    assert np.array_equal(bits(got[i]), want), (dt, lay, da, szs is None, i, ops[i])
            # ragged, with windows
            szs = [(int(rng.integers(8, 90)), int(rng.integers(8, 90))) for _ in range(n)]
            wins = [(1, 2, z[0] - 3, z[1] - 2) for z in szs]
            fmt = tensor_format(dt, lay, "mul", IMAGENET["mean"], IMAGENET["std"], da)
            eb = {"uint8": 1, "float32": 4, "float16": 2, "bfloat16": 2}[dt]
            C_ = 3 if da else full.shape[2]
            nb = [ww * wh * C_ * eb for (_, _, ww, wh) in wins]
            descs, foffs, fsizes, fb, poff = pack([f] * n, nb)
            fa = np.frombuffer(fb, np.uint8)
            out = np.zeros(poff + 16, np.uint8)
            codec.decode_blur_raw(fmt, descs, filter_codes("bicubic", n), op_codes(ops), rects(boxes), size_arr(szs), rects(wins),
                                  color_array(cols, n), blur_array(blurs, n), n, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                  out.ctypes.data, poff, 0)
            for i in range(n):
                want = to_tensor_ref(blur_entry_ref(full, cols[i], blurs[i], boxes[i], szs[i], 3, wins[i], ops[i]), dt, lay, "mul",
                                     IMAGENET["mean"], IMAGENET["std"], da)
                got = out[descs[i].offset: descs[i].offset + nb[i]].view(want.dtype).reshape(want.shape)
                assert np.array_equal(got, want), (dt, lay, da, "ragged", i, ops[i])


class DinoGaussianBlur:
    """DINO's utils.GaussianBlur: applied with probability p, radius uniform in [0.1, 2.0] from Python's random."""
    def __init__(self, p=0.5, radius_min=0.1, radius_max=2.0):
        self.prob, self.radius_min, self.radius_max = p, radius_min, radius_max

    def __call__(self, img):
        if not random.random() <= self.prob:
            return img
        return img.filter(ImageFilter.GaussianBlur(radius=random.uniform(self.radius_min, self.radius_max)))


class DinoSolarization:
    def __init__(self, p):
        self.p = p

    def __call__(self, img):
        return ImageOps.solarize(img) if random.random() < self.p else img


class MocoGaussianBlur:
    """MoCo v2's GaussianBlur([.1, 2.]): radius uniform in sigma from Python's random."""
    def __init__(self, sigma=(0.1, 2.0)):
        self.sigma = sigma

    def __call__(self, x):
        return x.filter(ImageFilter.GaussianBlur(radius=random.uniform(self.sigma[0], self.sigma[1])))


def _replay_view(rrc, img, cj, blur_p, sol_p, flip_first=True, blur_applied=None):
    """The draws of RRC -> flip -> ColorJitter p 0.8 -> gray p 0.2 -> blur -> solarize, in DINO's order: (box, op, colour, blur)."""
    import torch
    import torchvision.transforms as T
    i, j, h, w = T.RandomResizedCrop.get_params(img, rrc.scale, rrc.ratio)
    op = "mh" if torch.rand(1) < 0.5 else "tl"
    c = replay_jitter(cj)
    radius = random.uniform(0.1, 2.0) if random.random() <= blur_p else None
    thr = 128 if sol_p and random.random() < sol_p else None
    return (j, i, w, h), op, c, None if radius is None and thr is None else blur_params(radius, thr)


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_dino_views_replayed(codec, level):
    """DINO's two global views (224, bicubic; blur p 1.0, or blur p 0.1 then solarize p 0.2) and its local views (96, blur p
    0.5), drawn with torch's and Python's RNGs as DINO draws them, are bit-identical to DINO's PIL Compose."""
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
    views += [(lc, T.Compose([lc, flip_and_color, DinoGaussianBlur(p=0.5), normalize]), 0.5, 0.0)] * 4
    torch.manual_seed(82 + level)
    random.seed(82 + level)
    want = [[tf(Image.fromarray(im)) for _, tf, _, _ in views] for im in imgs]
    torch.manual_seed(82 + level)
    random.seed(82 + level)
    draws = [[_replay_view(rrc, Image.fromarray(im), cj, bp, sp) for rrc, _, bp, sp in views] for im in imgs]
    n_sol = n_blur = 0
    for v, (rrc, _, _, _) in enumerate(views):
        d = [dr[v] for dr in draws]
        s = rrc.size[0]
        got = codec.decode_tensor(files, [(s, s)] * len(files), [x[0] for x in d], [x[1] for x in d], torch.float32,
                                  mean=IMAGENET["mean"], std=IMAGENET["std"], filters="bicubic", colors=[x[2] for x in d],
                                  blurs=[x[3] for x in d]).cpu()
        assert torch.equal(got.view(torch.int32), torch.stack([w[v] for w in want]).view(torch.int32)), v
        n_sol += sum(x[3] is not None and x[3].solarize for x in d)
        n_blur += sum(x[3] is not None and x[3].radius[0] > 0 for x in d)
    assert n_blur > 20 and n_sol >= 1


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_moco_v2_replayed(codec, level):
    """A MoCo v2 batch (RRC 224 -> ColorJitter p 0.8 -> gray p 0.2 -> GaussianBlur p 0.5 -> flip): the flip after the blur
    commutes with it, so the replayed entries are bit-identical to the PIL Compose."""
    import torch
    import torchvision.transforms as T
    imgs = [synth.rgb(h, w, 2900 + k) for k, (w, h) in enumerate([(500, 375), (333, 500), (640, 427), (300, 300)] * 4)]
    files = [po.encode(level, im) for im in imgs]
    cj = T.ColorJitter(0.4, 0.4, 0.4, 0.1)
    rrc = T.RandomResizedCrop(224, scale=(0.2, 1.0))
    tf = T.Compose([rrc, T.RandomApply([cj], p=0.8), T.RandomGrayscale(p=0.2), T.RandomApply([MocoGaussianBlur([0.1, 2.0])], p=0.5),
                    T.RandomHorizontalFlip(), T.ToTensor(), T.Normalize(*IMAGENET.values())])
    torch.manual_seed(5 + level)
    random.seed(5 + level)
    want = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    torch.manual_seed(5 + level)
    random.seed(5 + level)
    boxes, ops, cols, blurs = [], [], [], []
    for im in imgs:
        i, j, h, w = T.RandomResizedCrop.get_params(Image.fromarray(im), rrc.scale, rrc.ratio)
        boxes.append((j, i, w, h))
        cols.append(replay_jitter(cj))
        blurs.append(blur_params(random.uniform(0.1, 2.0)) if not (0.5 < torch.rand(1)) else None)
        ops.append("mh" if torch.rand(1) < 0.5 else "tl")
    got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, torch.float32, mean=IMAGENET["mean"], std=IMAGENET["std"],
                              colors=cols, blurs=blurs).cpu()
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    assert sum(b is not None for b in blurs) >= 3


@gpu
def test_8k_frame_and_huge_radius(codec):
    """A whole 7680 x 4320 frame at radius 2, entries at radius 1e4 (box radius far wider than the image), 1 x 1, 1 x N and
    N x 1 entries."""
    import torch
    px = synth.rgb(4320, 7680, 61)
    f = codec.encode(1, [px])[0]
    b = blur_params(2.0, 128)
    got = codec.decode_tensor([f], None, None, None, torch.uint8, "hwc", blurs=[b]).cpu().numpy()[0]
    assert np.array_equal(got, pil_blur(px, b))
    small = synth.rgb(150, 230, 62)
    fs = po.encode(2, small)
    boxes = [(0, 0, 230, 150), (3, 4, 1, 1), (0, 7, 230, 1), (9, 0, 1, 150), (5, 5, 1, 9), (100, 20, 70, 40)]
    blurs = [blur_params(1e4), blur_params(1.7, 100), blur_params((3.0, 0.5)), blur_params(1e4, 128), blur_params(0.4), blur_params((1e4, 2.0))]
    check_u8(codec, [fs] * 6, [small] * 6, None, blurs, boxes, None, ["tl", "r90", "mh", "r270", "tl", "r90"])
    # tensor strips: a row, and a column turned into a row (its x passes run down the staged column)
    boxes, ops = [(0, 7, 150, 1), (9, 0, 1, 150), (3, 3, 1, 1)], ["tl", "r90", "r270"]
    for bl in ([blur_params(1e4), blur_params((1e4, 0.6), 128), blur_params((0.8, 1e4))],
               [blur_params((2.2, 0.0)), blur_params((0.0, 3.1)), blur_params(None, 40)]):
        got = codec.decode_tensor([fs] * 2, None, boxes[:2], ops[:2], torch.uint8, "hwc", blurs=bl[:2]).cpu().numpy()
        for i in range(2):
            assert np.array_equal(got[i], pil_blur(po.orient(ops[i], small[boxes[i][1]: boxes[i][1] + boxes[i][3],
                                                                          boxes[i][0]: boxes[i][0] + boxes[i][2]]), bl[i])), i
        got = codec.decode_tensor([fs], None, boxes[2:], ops[2:], torch.uint8, "hwc", blurs=bl[2:]).cpu().numpy()[0]
        assert np.array_equal(got, pil_blur(small[3:4, 3:4], bl[2]))


@gpu
def test_pipelined_chunks_device_resident(monkeypatch):
    """Sintel-like frames cut into at least 3 chunks on 2 lanes, files and output in device memory, uint8 and float32."""
    import torch
    frames = synth.sintel_batch(range(3000, 3008))
    for k, v in (("XPNGB_LAT_MAX_BLOCKS", "0"), ("XPNGB_PIPE_MIN_MPIX", "1"), ("XPNGB_PIPE_LANES", "2"), ("XPNGB_CHUNK_MPIX", "3")):
        monkeypatch.setenv(k, v)
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(199)
        n = len(frames)
        boxes = [(int(rng.integers(0, 900)), int(rng.integers(0, 500)), 1000, 500) for _ in range(n)]
        szs = [(224, 224) if k % 2 else None for k in range(n)]
        cols = [random_col(rng) if k % 3 else None for k in range(n)]
        blurs = [blur_params(float(rng.uniform(0.1, 2.0)), 128 if k % 2 else None) if k != 5 else None for k in range(n)]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for fmt, eb in ((None, 1), (tensor_format("float32", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True), 4)):
                nb = [(224 * 224 if z else b[2] * b[3]) * 3 * eb for z, b in zip(szs, boxes)]
                descs, foffs, fsizes, fb, poff = pack(files, nb)
                dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
                dout = torch.zeros(poff, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                zs = [z or (b[2], b[3]) for z, b in zip(szs, boxes)]
                cd.profile(True)
                cd.decode_blur_raw(fmt, descs, None, None, rects(boxes), size_arr(zs), None, color_array(cols, n), blur_array(blurs, n), n,
                                   dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dout.data_ptr(), poff, 1)
                rep = cd.profile_report()
                cd.profile(False)
                assert rep["k_blur"][1] >= 3 * 6, rep
                out = dout.cpu().numpy()
                for i in range(n):
                    px = blur_entry_ref(frames[i], cols[i], blurs[i], boxes[i], szs[i])
                    want = px if fmt is None else to_tensor_ref(px, "float32", "chw", "div", IMAGENET["mean"], IMAGENET["std"], True)
                    got = out[descs[i].offset: descs[i].offset + nb[i]]
                    assert np.array_equal(got, want.reshape(-1).view(np.uint8)), (lv, fmt is None, i)
    finally:
        cd.close()


@gpu
def test_null_and_empty_blurs_are_colour_decode(codec):
    """blurs == NULL and entries with radius (0, 0) and no solarize give the bytes of decode_color."""
    import torch
    imgs = [synth.rgb(300, 400, 1), synth.rgba(200, 260, 2), synth.rgb(123, 77, 3)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)]
    boxes = [(5, 6, 200, 150), (0, 0, 260, 200), (1, 1, 70, 100)]
    ops = ["r90", "mh", "tl"]
    cols = [col(b=1.3), None, col([3, 2, 1, 0], s=0.4, h=0.1)]
    empty = [None, blur_params(), blur_params(0.0, None)]
    base = codec.decode_resized(files, [(64, 48)] * 3, boxes, ops, "bicubic", [(2, 2, 50, 40)] * 3, colors=cols)
    for bl in (None, empty):
        nb = [50 * 40 * im.shape[2] for im in imgs]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.zeros(poff + 16, np.uint8)
        codec.decode_blur_raw(None, descs, filter_codes("bicubic", 3), op_codes(ops), rects(boxes), size_arr([(64, 48)] * 3),
                              rects([(2, 2, 50, 40)] * 3), color_array(cols, 3), blur_array(bl, 3), 3, fa.ctypes.data, len(fb), 0,
                              foffs, fsizes, out.ctypes.data, poff, 0)
        for i, w in enumerate(base):
            assert out[descs[i].offset: descs[i].offset + w.size].tobytes() == w.tobytes()
    t0 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, torch.bfloat16, "hwc", mean=IMAGENET["mean"], std=IMAGENET["std"],
                             drop_alpha=True, colors=cols)
    t1 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, torch.bfloat16, "hwc", mean=IMAGENET["mean"], std=IMAGENET["std"],
                             drop_alpha=True, colors=cols, blurs=empty)
    assert torch.equal(t0.view(torch.int16), t1.view(torch.int16))


@gpu
def test_blur_failures(codec):
    """Each refused input fails naming the entry, before anything is written."""
    px, pa = synth.rgb(100, 120, 5), synth.noise(90, 80, 6, channels=4)   # random alpha: the file keeps it
    f, fa_ = po.encode(1, px), po.encode(2, pa)
    assert po.decode(fa_).shape[2] == 4

    def call(b1, files=None, fmt=None):
        files = files or [f, f]
        nb = [100 * 120 * 4 * 4] * 2
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, 0xA5, np.uint8)
        err = None
        try:
            codec.decode_blur_raw(fmt, descs, None, None, None, None, None, None, blur_array([blur_params(1.0), b1], 2), 2, fa.ctypes.data,
                                  len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
        except RuntimeError as e:
            err = str(e)
        return err, out

    bad = [(blur_params(r), "radius") for r in (-0.1, -1e-300, math.inf, math.nan, 8388609.0, 8388608.6, 1e39, 1e300)]
    bad += [(blur_params((1.0, r)), "radius") for r in (-2.0, math.nan, 9e6)]
    b = blur_params(1.0, 128); b.solarize = 2; bad.append((b, "solarize"))
    bad.append((blur_params(None, math.nan), "NaN"))
    for b1, word in bad:
        err, out = call(b1)
        assert err is not None and "entry 1" in err and word in err and (out == 0xA5).all(), (list(b1.radius), err)
    for r in (RADIUS_MAX, 8388608.4):   # just below the bound: accepted, and equal to Pillow's result
        assert call(blur_params(r))[0] is None
        got = codec.decode_resized([f], [(120, 100)], blurs=[blur_params(r)])[0]
        assert np.array_equal(got, np.asarray(_pil(px).filter(ImageFilter.GaussianBlur(r))))
    for fmt in (None, tensor_format("float32")):   # solarize on an RGBA entry whose output keeps alpha
        err, out = call(blur_params(None, 128), [f, fa_], fmt)
        assert err is not None and "entry 1" in err and "alpha" in err and (out == 0xA5).all(), err
    assert call(blur_params(1.0, 128), [f, fa_], tensor_format("float32", drop_alpha=True))[0] is None
    assert call(blur_params(2.5), [f, fa_])[0] is None   # blur on RGBA is allowed
    assert call(blur_params(None, -math.inf))[0] is None
