"""Auto-augmented decode (xpngb_decode_augment / Codec.decode_resized and decode_tensor with augments): the 14 ops of
torchvision's transforms.autoaugment._apply_op on the PIL path, applied to each entry right after its op, byte-identical to
Pillow.  Entry i is tensor(solarize_i(blur_i(gray_i(jitter_i(augment_i(orient(op_i, window_i(resize_f(crop_i))))))))).

augment_ref() restates the C program (augment_params' output) in numpy: Pillow 12's ImagingTransformAffine with its three
NEAREST paths (ImagingScaleAffine, the 16.16 fixed-point affine_fixed, the double one) and the BILINEAR / BICUBIC filters of
ImagingGenericTransform, the rotate transposes, ImageEnhance's blends, SMOOTH, and the ImageOps LUTs.  The CPU tests pin it to
_apply_op on PIL images; on the GPU every output is compared with augment_ref or with torchvision itself."""
import math

import numpy as np
import pytest
from PIL import Image

from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import (AUG_KINDS, AUG_STEPS_MAX, _Augment, augment_array, augment_params, auto_augment_steps, blur_array,
                             color_array, filter_codes, op_codes, rand_augment_steps, rects, sizes as size_arr, tensor_format,
                             trivial_augment_wide_steps)
from test_blur_decode import blur_params, pil_blur, solarize_t
from test_color_decode import blend, col, color_ref, entry_ref, luma, random_col
from test_resampled_decode import FILTERS, pack
from test_tensor_decode import IMAGENET, bits, to_tensor_ref

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
K = AUG_KINDS
PATHS = {}   # Pillow code paths augment_ref went through, counted


# ---------------------------------------------------------------------------------------------------- the oracle

def _hit(path):
    PATHS[path] = PATHS.get(path, 0) + 1


def _seq(start, inc, n):
    """start, start + inc, ... (n values), each sum rounded as Pillow's running `xx += a[0]` is."""
    out = np.empty(n)
    v = float(start)
    for k in range(n):
        out[k] = v
        v += inc
    return out


def _x86_int(v):
    """C's (int) of a double as x86-64 computes it: truncation, INT_MIN for NaN and out of range."""
    v = np.asarray(v, dtype=np.float64)
    ok = (v > -2147483649.0) & (v < 2147483648.0)
    return np.where(ok, np.trunc(np.where(ok, v, 0)), -2147483648).astype(np.int64)


def _floor_int(v):   # Pillow's FLOOR
    v = np.asarray(v, dtype=np.float64)
    return np.where(v < 0, _x86_int(np.floor(v)), _x86_int(v))


def _nearest(px, a, fill):
    """Image.transform(AFFINE, a, NEAREST, fillcolor=fill) of an (h, w, c) uint8 array: Pillow's three NEAREST paths."""
    h, w = px.shape[:2]
    out = np.empty_like(px)
    out[:] = np.asarray(fill, np.uint8)[: px.shape[2]]
    if a[1] == 0 and a[3] == 0:   # ImagingScaleAffine
        _hit("scale")
        xs, ys = _seq(a[2] + a[0] * 0.5, a[0], w), _seq(a[5] + a[4] * 0.5, a[4], h)
        X, Y = np.meshgrid(xs, ys)
    elif all(abs(x * a[0] + y * a[1] + a[2]) < 32768.0 and abs(x * a[3] + y * a[4] + a[5]) < 32768.0
             for x, y in ((0, 0), (w, h), (0, h), (w, 0))):   # affine_fixed
        _hit("fixed")
        fix = [int(_floor_int(v * 65536.0 + 0.5)) for v in (a[0], a[1], a[2] + a[0] * 0.5 + a[1] * 0.5, a[3], a[4],
                                                             a[5] + a[3] * 0.5 + a[4] * 0.5)]
        x, y = np.meshgrid(np.arange(w, dtype=np.int64), np.arange(h, dtype=np.int64))
        wrap = lambda v: ((v + (1 << 31)) % (1 << 32)) - (1 << 31)
        xi = wrap(fix[2] + y * fix[1] + x * fix[0]) >> 16
        yi = wrap(fix[5] + y * fix[4] + x * fix[3]) >> 16
        ok = (xi >= 0) & (xi < w) & (yi >= 0) & (yi < h)
        out[ok] = px[yi[ok], xi[ok]]
        return out
    else:   # the double path: running sums along each row, row starts by running sums down the image
        _hit("double")
        x0s, y0s = _seq(a[2] + a[1] * 0.5 + a[0] * 0.5, a[1], h), _seq(a[5] + a[4] * 0.5 + a[3] * 0.5, a[4], h)
        X, Y = np.empty((h, w)), np.empty((h, w))
        xx, yy = x0s.copy(), y0s.copy()
        for k in range(w):
            X[:, k], Y[:, k] = xx, yy
            xx += a[0]
            yy += a[3]
    ok = (X >= 0) & (X < w) & (Y >= 0) & (Y < h)
    out[ok] = px[np.trunc(Y[ok]).astype(np.int64), np.trunc(X[ok]).astype(np.int64)]
    return out


def _generic(px, a, resample, fill):
    """ImagingGenericTransform with Pillow's bilinear or bicubic filter (Geometry.c), every double operation on its own."""
    _hit("bilinear" if resample == 2 else "bicubic")
    h, w, c = px.shape
    x, y = np.meshgrid(np.arange(w) + 0.5, np.arange(h) + 0.5)
    xin = a[0] * x + a[1] * y + a[2]
    yin = a[3] * x + a[4] * y + a[5]
    ok = (xin >= 0.0) & (xin < w) & (yin >= 0.0) & (yin < h)
    out = np.empty_like(px)
    out[:] = np.asarray(fill, np.uint8)[:c]
    xin, yin = xin[ok] - 0.5, yin[ok] - 0.5
    xf, yf = _floor_int(xin), _floor_int(yin)
    dx, dy = (xin - xf)[:, None], (yin - yf)[:, None]
    p = px.astype(np.float64)

    def row(yr, xs):   # the samples of row yr at columns xs, clipped (XCLIP / YCLIP)
        return [p[np.clip(yr, 0, h - 1), np.clip(xx, 0, w - 1)] for xx in xs]

    if resample == 2:
        lin = lambda u, v, d: u + (v - u) * d
        r0 = row(yf, (xf, xf + 1))
        v1 = lin(r0[0], r0[1], dx)
        r1 = row(yf + 1, (xf, xf + 1))
        v2 = np.where(((yf + 1 >= 0) & (yf + 1 < h))[:, None], lin(r1[0], r1[1], dx), v1)
        v = lin(v1, v2, dy)
        out[ok] = v.astype(np.uint8)
        return out

    def cub(v1, v2, v3, v4, d):
        p1, p2, p3, p4 = v2, -v1 + v3, 2 * (v1 - v2) + v3 - v4, -v1 + v2 - v3 + v4
        return p1 + d * (p2 + d * (p3 + d * p4))

    xm, ym = xf - 1, yf - 1
    cols = (xm, xm + 1, xm + 2, xm + 3)
    vs = [cub(*row(ym, cols), dx)]
    for k in (1, 2, 3):
        inside = ((ym + k >= 0) & (ym + k < h))[:, None]
        vs.append(np.where(inside, cub(*row(ym + k, cols), dx), vs[-1]))
    v = cub(*vs, dy)
    out[ok] = np.where(v <= 0.0, 0, np.where(v >= 255.0, 255, np.clip(v, 0, 255).astype(np.int64))).astype(np.uint8)
    return out


def transpose_ref(px, op):
    return np.ascontiguousarray(po.orient(op, px))


def smooth_ref(px):
    """ImageFilter.SMOOTH (3 x 3, 1 1 1 / 1 5 1 / 1 1 1, divisor 13): borders copied, round-half-up of the weighted mean."""
    h, w = px.shape[:2]
    out = px.copy()
    if h < 3 or w < 3:
        return out
    p = px.astype(np.int64)
    s = 4 * p[1:-1, 1:-1]
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            s = s + p[1 + dy: h - 1 + dy, 1 + dx: w - 1 + dx]
    out[1:-1, 1:-1] = (s + 6) // 13
    return out


def equalize_lut(ch):
    """ImageOps.equalize's LUT of one channel: Python's integer rule."""
    hist = np.bincount(ch.reshape(-1), minlength=256)
    nz = hist[hist > 0]
    if len(nz) <= 1:
        return np.arange(256)
    step = (int(nz.sum()) - int(nz[-1])) // 255
    if not step:
        return np.arange(256)
    n = step // 2 + np.concatenate([[0], np.cumsum(hist)[:-1]])
    return np.minimum(n // step, 255)   # Image.point clips the LUT to bytes


def autocontrast_lut(ch):
    hist = np.bincount(ch.reshape(-1), minlength=256)
    nz = np.nonzero(hist)[0]
    lo, hi = int(nz[0]), int(nz[-1])
    if hi <= lo:
        return np.arange(256)
    scale = 255.0 / (hi - lo)
    offset = -lo * scale
    return np.array([min(max(int(ix * scale + offset), 0), 255) for ix in range(256)])


def augment_ref(px, aug):
    """The (h, w, 3) uint8 array px after the program aug (an xpngb_augment)."""
    out = px.copy()
    for s in aug.step[: aug.nsteps]:
        kind, rgb = s.kind, out[..., :3]
        if kind == K["affine"]:
            a, fill = list(s.data), list(s.fill)
            out = _nearest(out, a, fill) if s.arg == 0 else _generic(out, a, s.arg, fill)
        elif kind == K["transpose"]:
            _hit("transpose")
            out = transpose_ref(out, ALL_OPS[s.arg])
        elif kind in (K["brightness"], K["color"], K["contrast"]):
            d = 0 if kind == K["brightness"] else luma(rgb)[..., None] if kind == K["color"] else int(int(luma(rgb).sum()) / luma(rgb).size + 0.5)
            out[..., :3] = blend(d, rgb, s.value)
        elif kind == K["sharpness"]:
            out[..., :3] = blend(smooth_ref(rgb).astype(np.int64), rgb, s.value)
        else:
            if kind == K["posterize"]:
                lut = [np.arange(256) & ~((1 << (8 - s.arg)) - 1) & 255] * 3
            elif kind == K["solarize"]:
                t = solarize_t(s.value)
                lut = [np.where(np.arange(256) < t, np.arange(256), 255 - np.arange(256))] * 3
            elif kind == K["invert"]:
                lut = [255 - np.arange(256)] * 3
            elif kind == K["equalize"]:
                lut = [equalize_lut(rgb[..., c]) for c in range(3)]
            else:
                lut = [autocontrast_lut(rgb[..., c]) for c in range(3)]
            for c in range(3):
                out[..., c] = np.asarray(lut[c], np.uint8)[rgb[..., c]]
    return out


def _pil(px):
    return Image.fromarray(px, "RGB")


def apply_op_pil(px, steps, interpolation, fill):
    """torchvision's _apply_op on the PIL image of px, step by step."""
    from torchvision.transforms import InterpolationMode
    from torchvision.transforms.autoaugment import _apply_op
    img = _pil(px)
    for name, m in steps:
        img = _apply_op(img, name, m, interpolation=InterpolationMode(interpolation), fill=fill)
    return np.asarray(img)


# ---------------------------------------------------------------------------------------------------- oracle against PIL (CPU)

def _spaces(w, h):
    import torchvision.transforms as T
    yield "rand", T.RandAugment()._augmentation_space(31, (h, w))
    yield "trivial", T.TrivialAugmentWide()._augmentation_space(31)
    yield "auto", T.AutoAugment()._augmentation_space(10, (h, w))


def every_op(w, h):
    """(op_name, magnitude) for every op x every magnitude bin of the three augmentation spaces, both signs."""
    seen = []
    for _, space in _spaces(w, h):
        for name, (mags, signed) in space.items():
            for m in ([float(v) for v in mags] if mags.ndim else [0.0]):
                for sg in ((1.0, -1.0) if signed else (1.0,)):
                    if (name, sg * m) not in seen:
                        seen.append((name, sg * m))
    return seen


GEOMETRIC = ("ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate")
SIZES = [(1, 1), (1, 9), (9, 1), (2, 9), (9, 2), (16, 16), (23, 31), (40, 40)]


@pytest.mark.parametrize("hw", SIZES + [(2, 40000)])
def test_restatement_matches_torchvision(hw):
    """augment_ref(augment_params(step)) equals _apply_op on the PIL image for every op at every bin of the three spaces,
    both signs, NEAREST / BILINEAR / BICUBIC, fill None and non-zero.  The 2 x 40000 image (NEAREST geometry only) takes
    Pillow's double path."""
    h, w = hw
    rng = np.random.default_rng(h * 100003 + w)
    px = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    cases = 0
    for name, m in every_op(w, h):
        for interp in ("nearest", "bilinear", "bicubic"):
            for fill in (None, (7, 200, 33.9)):
                if w > 1000 and (interp != "nearest" or name not in GEOMETRIC):
                    continue
                if name not in GEOMETRIC and (interp != "nearest" or fill is not None):
                    continue   # only the warps read them
                st = [(name, m)]
                want = apply_op_pil(px, st, interp, fill)
                assert np.array_equal(augment_ref(px, augment_params(st, (w, h), interp, fill)), want), (hw, name, m, interp, fill)
                cases += 1
    assert cases > (100 if w > 1000 else 900)


def test_paths_are_reached():
    """All three NEAREST paths, both generic filters, and the 180 and square 90 / 270 rotate fast paths (TrivialAugmentWide's
    rotate bin 20 is exactly 90.0) are reached."""
    PATHS.clear()
    px = np.random.default_rng(5).integers(0, 256, (2, 40000, 3), dtype=np.uint8)
    augment_ref(px, augment_params([("Rotate", 10.0)], (40000, 2)))
    sq = np.random.default_rng(6).integers(0, 256, (24, 24, 3), dtype=np.uint8)
    for st in ([("TranslateX", 3.0)], [("ShearY", 0.2)], [("Rotate", 15.0)]):
        for interp in ("nearest", "bilinear", "bicubic"):
            augment_ref(sq, augment_params(st, (24, 24), interp))
    assert all(PATHS.get(p, 0) > 0 for p in ("scale", "fixed", "double", "bilinear", "bicubic")), PATHS
    import torchvision.transforms as T
    m90 = float(T.TrivialAugmentWide()._augmentation_space(31)["Rotate"][0][20])
    assert m90 == 90.0
    for m, op in ((m90, "r270"), (-m90, "r90"), (180.0, "mvh"), (-180.0, "mvh")):
        a = augment_params([("Rotate", m)], (24, 24))
        assert a.nsteps == 1 and a.step[0].kind == K["transpose"] and ALL_OPS[a.step[0].arg] == op, m
        assert np.array_equal(augment_ref(sq, a), apply_op_pil(sq, [("Rotate", m)], "nearest", None))
    assert augment_params([("Rotate", m90)], (24, 20)).step[0].kind == K["affine"]   # not square: the matrix
    assert augment_params([("Rotate", 0.0)], (24, 20)).nsteps == 0 and augment_params([("Rotate", 360.0)], (3, 3)).nsteps == 0


def _replays(n_draws, seed):
    import torch
    import torchvision.transforms as T
    from torchvision.transforms import AutoAugmentPolicy as P, InterpolationMode as IM
    mods = [T.RandAugment(num_ops=k, magnitude=mg, interpolation=ip, fill=fl)
            for k, mg, ip, fl in ((1, 9, IM.NEAREST, None), (2, 9, IM.BILINEAR, None), (3, 30, IM.BICUBIC, 17), (2, 0, IM.NEAREST, [3, 9, 250]))]
    mods += [T.TrivialAugmentWide(interpolation=ip, fill=fl) for ip, fl in ((IM.NEAREST, None), (IM.BILINEAR, 128), (IM.BICUBIC, None))]
    mods += [T.AutoAugment(p, ip) for p in (P.IMAGENET, P.CIFAR10, P.SVHN) for ip in (IM.NEAREST, IM.BILINEAR)]
    replay = {T.RandAugment: rand_augment_steps, T.TrivialAugmentWide: trivial_augment_wide_steps, T.AutoAugment: auto_augment_steps}
    rng = np.random.default_rng(seed)
    for k in range(n_draws):
        mod = mods[k % len(mods)]
        h, w = [(16, 16), (20, 24), (9, 13), (32, 32)][k % 4]
        px = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if k % 5 == 0:   # flat regions: degenerate histograms and exact blends
            px = np.repeat(np.repeat(px[::4, ::4], 4, 0), 4, 1)[:h, :w].copy()
        torch.manual_seed(seed * 1000 + k)
        want = np.asarray(mod(_pil(px)))
        torch.manual_seed(seed * 1000 + k)
        yield mod, px, want, replay[type(mod)](mod, (w, h))


def test_replay_matches_torchvision():
    """Seeded RandAugment (several num_ops and magnitudes), TrivialAugmentWide and AutoAugment (IMAGENET, CIFAR10, SVHN)
    forwards on PIL equal augment_ref of the replayed program, over hundreds of draws."""
    steps = 0
    for mod, px, want, aug in _replays(650, 1):
        assert np.array_equal(augment_ref(px, aug), want), (mod, [(s.kind, s.arg, s.value) for s in aug.step[: aug.nsteps]])
        steps += aug.nsteps
    assert steps > 500


@pytest.mark.parametrize("op", ALL_OPS)
def test_pointwise_steps_commute_with_the_op(op):
    """The histogram, LUT, blend and SMOOTH steps give the same result under every op: they can run on staged tensor
    entries as they sit."""
    rng = np.random.default_rng(ALL_OPS.index(op) + 40)
    kinds = [("Brightness", 0.4), ("Color", -0.7), ("Contrast", 0.55), ("Sharpness", 0.9), ("Sharpness", -0.6), ("Posterize", 3.0),
             ("Solarize", 99.6), ("AutoContrast", 0.0), ("Equalize", 0.0), ("Invert", 0.0)]
    for k in range(30):
        h, w = int(rng.integers(1, 30)), int(rng.integers(1, 30))
        x = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        st = [kinds[k % len(kinds)], kinds[(k * 7 + 3) % len(kinds)]]
        a = augment_params(st, (w, h))
        assert np.array_equal(augment_ref(transpose_ref(x, op), a), transpose_ref(augment_ref(x, a), op)), (op, st)


def test_smooth_integer_form():
    """SMOOTH's interior equals (S + 6) // 13 of the weighted sum S on many random and blocky images (Sharpness at factor 0
    is SMOOTH itself), borders and images with a side below 3 are copied."""
    from PIL import ImageFilter
    rng = np.random.default_rng(7)
    for k in range(300):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        x = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if k % 3 == 0:
            x = (x // 64 * 85).astype(np.uint8)
        assert np.array_equal(smooth_ref(x), np.asarray(_pil(x).filter(ImageFilter.SMOOTH))), (h, w)


def test_degenerate_histograms():
    """Single colour, one non-empty bin per channel, equalize's step 0, and hi <= lo give the identity LUT, as Pillow."""
    from PIL import ImageOps
    rng = np.random.default_rng(8)
    imgs = [np.full((7, 9, 3), 77, np.uint8), np.dstack([np.full((5, 5), v, np.uint8) for v in (0, 128, 255)])]
    few = np.full((20, 20, 3), 200, np.uint8)
    few[0, :3] = 10    # step = (400 - 397) // 255 == 0
    imgs += [few, rng.integers(0, 2, (1, 1, 3), dtype=np.uint8), rng.integers(100, 102, (30, 3, 3), dtype=np.uint8)]
    big = rng.integers(0, 256, (300, 300, 3), dtype=np.uint8)   # lut values above 255 before Image.point clips them
    imgs.append(big)
    for x in imgs:
        for name, fn in (("Equalize", ImageOps.equalize), ("AutoContrast", ImageOps.autocontrast)):
            assert np.array_equal(augment_ref(x, augment_params([(name, 0.0)], x.shape[1::-1])), np.asarray(fn(_pil(x)))), (name, x.shape)
    assert np.array_equal(equalize_lut(few[..., 0]), np.arange(256))


def test_augment_params_fields():
    import ctypes as C
    assert C.sizeof(_Augment) == 8 + AUG_STEPS_MAX * 72
    a = augment_params([("TranslateY", -7.9), ("Posterize", 5.7), ("Solarize", 12.5), ("Sharpness", -0.3)], (50, 40), "bicubic", 3.9)
    assert a.nsteps == 4 and a.step[0].kind == K["affine"] and a.step[0].arg == 3 and list(a.step[0].fill) == [3, 3, 3, 0]
    assert list(a.step[0].data) == [1.0, 0.0, 0.0, -0.0, 1.0, 7.0]   # int(-7.9) = -7
    assert a.step[1].arg == 5 and a.step[2].value == 12.5 and a.step[3].value == 0.7
    assert augment_params([("Identity", 0.0)] * 20, (5, 5)).nsteps == 0
    for bad in (lambda: augment_params([("Cutout", 1.0)], (5, 5)), lambda: augment_params([("Invert", 0.0)] * 9, (5, 5)),
                lambda: augment_params([], (5, 5), "lanczos"), lambda: augment_params([], (5, 5), fill=(1, 2)),
                lambda: augment_params([], (5, 5), fill=300)):
        with pytest.raises(ValueError):
            bad()
    arr = augment_array([None, a], 2)
    assert arr[0].nsteps == 0 and arr[1].nsteps == 4


def test_pillow_refuses_rgba():
    from PIL import ImageOps
    im = Image.fromarray(np.zeros((4, 4, 4), np.uint8), "RGBA")
    for fn in (ImageOps.invert, ImageOps.equalize, ImageOps.autocontrast, lambda i: ImageOps.posterize(i, 3)):
        with pytest.raises(OSError):
            fn(im)


# ---------------------------------------------------------------------------------------------------- augmented decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


def aug_entry_ref(full, aug, rect=None, size=None, filt=2, win=None, op=None, c=None, b=None):
    """Pillow's chain for one entry: crop, resize, window, op, then (RGB) augment, colour, blur and solarize."""
    px = entry_ref(full, None, rect, size, filt, win, op)
    if aug is not None and aug.nsteps:
        px = augment_ref(np.ascontiguousarray(px[..., :3]), aug)
    px = px if c is None else color_ref(px, c)
    return pil_blur(px, b)


def _hw(full, rect, size, win, op):
    w, h = (win[2], win[3]) if win else size if size else (rect[2], rect[3]) if rect else full.shape[1::-1]
    return (w, h) if op in ("r90", "r270") else (h, w)


def run(cd, files, fulls, augs, boxes=None, szs=None, ops=None, filters=None, wins=None, cols=None, blurs=None, fmt=None, dt="uint8",
        lay="hwc", da=False, scale="div", mean=(0, 0, 0, 0), std=(1, 1, 1, 1)):
    """decode_augment_raw against aug_entry_ref (and to_tensor_ref for tensor output)."""
    n = len(files)
    g = lambda v, i: None if v is None else v[i]
    eb = {"uint8": 1, "float32": 4, "float16": 2, "bfloat16": 2}[dt]
    hw = [_hw(fulls[i], g(boxes, i), g(szs, i), g(wins, i), g(ops, i)) for i in range(n)]
    ch = [3 if da else fulls[i].shape[2] for i in range(n)]
    nb = [h * w * ch[i] * eb for i, (h, w) in enumerate(hw)]
    descs, foffs, fsizes, fb, poff = pack(files, nb)
    fa = np.frombuffer(fb, np.uint8)
    out = np.zeros(poff + 16, np.uint8)
    cd.decode_augment_raw(fmt, descs, None if filters is None else filter_codes(filters, n), None if ops is None else op_codes(ops),
                          None if boxes is None else rects(boxes), None if szs is None else size_arr(szs),
                          None if wins is None else rects(wins), None if cols is None else color_array(cols, n),
                          None if blurs is None else blur_array(blurs, n), augment_array(augs, n), n, fa.ctypes.data, len(fb), 0,
                          foffs, fsizes, out.ctypes.data, poff, 0)
    for i in range(n):
        px = aug_entry_ref(fulls[i], augs[i], g(boxes, i), g(szs, i), 2 if filters is None else filters[i], g(wins, i), g(ops, i),
                           g(cols, i), g(blurs, i))
        if fmt is None:
            want = px
        else:
            want = to_tensor_ref(px, dt, lay, scale, mean, std, da)
        got = out[descs[i].offset: descs[i].offset + nb[i]]
        assert np.array_equal(got, np.ascontiguousarray(want).reshape(-1).view(np.uint8)), \
            (i, g(ops, i), [(s.kind, s.arg, s.value, list(s.data)) for s in augs[i].step[: augs[i].nsteps]] if augs[i] else None)


def matrix(w, h):
    """Each op alone at each bin of the three spaces, both signs; the warps under each interpolation, fill None and not."""
    progs = []
    for k, (name, m) in enumerate(every_op(w, h)):
        for interp in (("nearest", "bilinear", "bicubic") if name in GEOMETRIC else ("nearest",)):
            progs.append(augment_params([(name, m)], (w, h), interp, None if k % 2 else (250, 3, 77)))
    return progs


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_coverage_matrix(codec, level):
    """Every op at every bin x every interpolation on uint8 crops under all seven ops (square and not: quarter turns swap
    the output), resized entries with the five filters and windows, and whole images."""
    rng = np.random.default_rng(300 + level)
    full = synth.rgb(230, 310, level + 60)
    f = po.encode(level, full)
    for cw, chh in ((48, 48), (61, 37)):
        progs = []
        ops = []
        for j, op in enumerate(ALL_OPS):
            w, h = (chh, cw) if op in ("r90", "r270") else (cw, chh)
            ps = matrix(w, h)
            progs += ps[j::7 if cw != chh else 1][: 400 if cw == chh else 90]
            ops += [op] * len(ps[j::7 if cw != chh else 1][: 400 if cw == chh else 90])
        n = len(progs)
        boxes = [(int(x), int(y), cw, chh) for x, y in zip(rng.integers(0, 310 - cw, n), rng.integers(0, 230 - chh, n))]
        run(codec, [f] * n, [full] * n, progs, boxes, None, ops)
    # resized, the five filters, windows (the program is built for the window's size after the op)
    n = 70
    szs = [(int(rng.integers(20, 90)), int(rng.integers(20, 90))) for _ in range(n)]
    wins = [(1, 2, z[0] - 3, z[1] - 4) for z in szs]
    ops = [ALL_OPS[j % 7] for j in range(n)]
    boxes = [(5, 9, 200, 150)] * n
    progs = []
    for j in range(n):
        w, h = (wins[j][3], wins[j][2]) if ops[j] in ("r90", "r270") else (wins[j][2], wins[j][3])
        eo = every_op(w, h)
        progs.append(augment_params([eo[(j * 37 + t * 11) % len(eo)] for t in range(3)], (w, h), ("nearest", "bilinear", "bicubic")[j % 3],
                                    (9, 8, 7)))
    run(codec, [f] * n, [full] * n, progs, boxes, szs, ops, [FILTERS[j % 5] for j in range(n)], wins)
    whole = [augment_params([("Rotate", 33.0), ("Equalize", 0.0)], (310, 230), "bilinear"), augment_params([("ShearX", 0.3)], (310, 230))]
    run(codec, [f] * 2, [full] * 2, whole)


TENSOR_FORMATS = [(dt, lay, da) for dt in ("float32", "float16", "bfloat16", "uint8") for lay in ("chw", "hwc") for da in (False, True)]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_tensor_formats(codec, level):
    """Every tensor format under every op: tensor entries sit before the op in scratch, so their warps map coordinates
    through it; RGBA files with drop_alpha are augmented as their RGB image."""
    rng = np.random.default_rng(400 + level)
    for im in (synth.rgb(200, 260, level + 70), synth.rgba(180, 240, level + 71)):
        f = po.encode(level, im)
        full = po.decode(f)
        a = full.shape[2] == 4
        for t, (dt, lay, da) in enumerate(TENSOR_FORMATS):
            if a and not da:
                continue
            n = 21
            ops = [ALL_OPS[j % 7] for j in range(n)]
            szs = [(40, 40) if j % 3 else (52, 33) for j in range(n)] if t % 2 else None
            boxes = [(int(rng.integers(0, 120)), int(rng.integers(0, 100)), 52, 33 if j % 2 else 52) for j in range(n)]
            progs = []
            for j in range(n):
                w, h = szs[j] if szs else boxes[j][2:]
                if ops[j] in ("r90", "r270"):
                    w, h = h, w
                eo = every_op(w, h)
                steps = [eo[int(rng.integers(len(eo)))] for _ in range(int(rng.integers(1, 4)))]
                steps[0] = (GEOMETRIC[j % 5], [0.3, -0.3, 7.0, -5.0, 41.0][j % 5])   # a warp in every entry
                progs.append(augment_params(steps, (w, h), ("nearest", "bilinear", "bicubic")[j % 3]))
            fmt = tensor_format(dt, lay, "div", IMAGENET["mean"], IMAGENET["std"], da)
            run(codec, [f] * n, [full] * n, progs, boxes, szs, ops, None, None, fmt=fmt, dt=dt, lay=lay, da=da,
                mean=IMAGENET["mean"], std=IMAGENET["std"])


def _preset_train(policy, level, seed, n=16):
    """A replayed ClassificationPresetTrain (RandomResizedCrop 224 bilinear, flip, policy, PILToTensor, ToDtype(scale),
    Normalize) against torchvision's PIL path, bit for bit."""
    import torch
    import torchvision.transforms.v2 as T2
    import torchvision.transforms as T
    imgs = [synth.rgb(h, w, seed + k) for k, (w, h) in enumerate([(500, 375), (333, 500), (640, 427), (300, 300)] * (n // 4))]
    files = [po.encode(level, im) for im in imgs]
    rrc = T.RandomResizedCrop(224, interpolation=T.InterpolationMode.BILINEAR, antialias=True)
    tf = T2.Compose([rrc, T.RandomHorizontalFlip(0.5), policy, T2.PILToTensor(), T2.ToDtype(torch.float, scale=True),
                     T2.Normalize(IMAGENET["mean"], IMAGENET["std"])])
    torch.manual_seed(seed)
    want = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    torch.manual_seed(seed)
    replay = {T.RandAugment: rand_augment_steps, T.TrivialAugmentWide: trivial_augment_wide_steps, T.AutoAugment: auto_augment_steps}
    boxes, ops, augs = [], [], []
    for im in imgs:
        i, j, h, w = T.RandomResizedCrop.get_params(Image.fromarray(im), rrc.scale, rrc.ratio)
        boxes.append((j, i, w, h))
        ops.append("mh" if torch.rand(1) < 0.5 else "tl")
        augs.append(replay[type(policy)](policy, (224, 224)))
    return files, boxes, ops, augs, want


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_classification_preset_train_replayed(codec, level):
    """ClassificationPresetTrain with TrivialAugmentWide (bilinear), RandAugment and AutoAugment: one decode_tensor call
    per batch is bit-identical to torchvision's PIL path."""
    import torch
    import torchvision.transforms as T
    from torchvision.transforms import InterpolationMode as IM
    steps = 0
    for k, pol in enumerate((T.TrivialAugmentWide(interpolation=IM.BILINEAR), T.RandAugment(2, 9, interpolation=IM.BILINEAR),
                             T.AutoAugment(T.AutoAugmentPolicy.IMAGENET, IM.BILINEAR), T.TrivialAugmentWide())):
        for rep in range(3):
            files, boxes, ops, augs, want = _preset_train(pol, level, 700 + 50 * k + 10 * rep + level)
            got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, torch.float32, scale="mul",
                                      mean=IMAGENET["mean"], std=IMAGENET["std"], augments=augs).cpu()
            assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (k, rep)
            steps += sum(a.nsteps for a in augs)
    assert steps > 100


@gpu
def test_with_colour_and_blur(codec):
    """Augment, colour and blur in one call (the blur's ping-pong starts from whichever buffer the program ended in), uint8
    and tensor, every op."""
    rng = np.random.default_rng(9)
    full = synth.rgb(240, 320, 90)
    f = po.encode(2, full)
    n = 28
    ops = [ALL_OPS[j % 7] for j in range(n)]
    boxes = [(int(rng.integers(0, 200)), int(rng.integers(0, 150)), 70, 50) for _ in range(n)]
    progs = []
    for j in range(n):
        w, h = (50, 70) if ops[j] in ("r90", "r270") else (70, 50)
        eo = every_op(w, h)
        progs.append(augment_params([eo[int(rng.integers(len(eo)))] for _ in range(1 + j % 3)], (w, h), ("nearest", "bilinear")[j % 2]))
    cols = [random_col(rng) if j % 2 else None for j in range(n)]
    blurs = [blur_params(float(rng.uniform(0.1, 2.0)), 128 if j % 3 else None) if j % 4 else None for j in range(n)]
    run(codec, [f] * n, [full] * n, progs, boxes, None, ops, cols=cols, blurs=blurs)
    fmt = tensor_format("float32", "chw", "div", IMAGENET["mean"], IMAGENET["std"])
    run(codec, [f] * n, [full] * n, progs, boxes, None, ops, cols=cols, blurs=blurs, fmt=fmt, dt="float32", lay="chw",
        mean=IMAGENET["mean"], std=IMAGENET["std"])


@gpu
def test_degenerate_and_8k_entries(codec):
    """Single-colour entries and equalize's step 0 (identity LUTs), and a whole 7680 x 4320 frame's histograms."""
    import torch
    flat = np.full((64, 64, 3), 91, np.uint8)
    two = np.full((64, 64, 3), 200, np.uint8)
    two[0, :3] = 10
    files = [codec.encode(1, [x])[0] for x in (flat, two)]
    progs = [augment_params([(s, 0.0)], (64, 64)) for s in ("Equalize", "AutoContrast")]
    for x, fl in zip((flat, two), files):
        run(codec, [fl] * 2, [x] * 2, progs)
    px = synth.rgb(4320, 7680, 61)
    f = codec.encode(1, [px])[0]
    for name in ("Equalize", "AutoContrast"):
        a = augment_params([(name, 0.5)], (7680, 4320))
        got = codec.decode_tensor([f], None, None, None, torch.uint8, "hwc", augments=[a]).cpu().numpy()[0]
        assert np.array_equal(got, augment_ref(px, a)), name


@gpu
def test_pipelined_chunks_device_resident(monkeypatch):
    """Sintel-like frames cut into at least 3 chunks on 2 lanes, files and output in device memory, uint8 and float32."""
    import torch
    frames = synth.sintel_batch(range(3100, 3108))
    for k, v in (("XPNGB_LAT_MAX_BLOCKS", "0"), ("XPNGB_PIPE_MIN_MPIX", "1"), ("XPNGB_PIPE_LANES", "2"), ("XPNGB_CHUNK_MPIX", "3")):
        monkeypatch.setenv(k, v)
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(299)
        n = len(frames)
        boxes = [(int(rng.integers(0, 900)), int(rng.integers(0, 500)), 1000, 500) for _ in range(n)]
        szs = [(224, 224) if k % 2 else (1000, 500) for k in range(n)]
        progs = [augment_params([("Rotate", 20.0 + k), ("Equalize", 0.0), ("ShearX", -0.2)], szs[k], "bilinear") for k in range(n)]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for fmt, eb in ((None, 1), (tensor_format("float32", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True), 4)):
                nb = [z[0] * z[1] * 3 * eb for z in szs]
                descs, foffs, fsizes, fb, poff = pack(files, nb)
                dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
                dout = torch.zeros(poff, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                cd.profile(True)
                cd.decode_augment_raw(fmt, descs, None, None, rects(boxes), size_arr(szs), None, None, None, augment_array(progs, n), n,
                                      dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dout.data_ptr(), poff, 1)
                rep = cd.profile_report()
                cd.profile(False)
                assert rep["k_aug_pix"][1] >= 3 * 2 and rep["k_aug_lut_build"][1] >= 3, rep
                out = dout.cpu().numpy()
                for i in range(n):
                    px = aug_entry_ref(frames[i], progs[i], boxes[i], szs[i])
                    want = px if fmt is None else to_tensor_ref(px, "float32", "chw", "div", IMAGENET["mean"], IMAGENET["std"], True)
                    assert np.array_equal(out[descs[i].offset: descs[i].offset + nb[i]], want.reshape(-1).view(np.uint8)), (lv, fmt is None, i)
    finally:
        cd.close()


@gpu
def test_null_and_empty_programs_are_blur_decode(codec):
    """augs == NULL and entries with no step give the bytes of decode_blur."""
    import torch
    imgs = [synth.rgb(300, 400, 1), synth.rgba(200, 260, 2), synth.rgb(123, 77, 3)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7), imgs)]
    boxes = [(5, 6, 200, 150), (0, 0, 260, 200), (1, 1, 70, 100)]
    ops = ["r90", "mh", "tl"]
    cols = [col(b=1.3), None, col([3, 2, 1, 0], s=0.4, h=0.1)]
    blurs = [blur_params(1.1), None, blur_params(0.7, 128)]
    base = codec.decode_resized(files, [(64, 48)] * 3, boxes, ops, "bicubic", [(2, 2, 50, 40)] * 3, colors=cols, blurs=blurs)
    for au in (None, [None, augment_params([], (1, 1)), _Augment()]):
        nb = [50 * 40 * im.shape[2] for im in imgs]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.zeros(poff + 16, np.uint8)
        codec.decode_augment_raw(None, descs, filter_codes("bicubic", 3), op_codes(ops), rects(boxes), size_arr([(64, 48)] * 3),
                                 rects([(2, 2, 50, 40)] * 3), color_array(cols, 3), blur_array(blurs, 3), augment_array(au, 3), 3,
                                 fa.ctypes.data, len(fb), 0, foffs, fsizes, out.ctypes.data, poff, 0)
        for i, w in enumerate(base):
            assert out[descs[i].offset: descs[i].offset + w.size].tobytes() == w.tobytes()
    kw = dict(dtype=torch.bfloat16, layout="hwc", mean=IMAGENET["mean"], std=IMAGENET["std"], drop_alpha=True, colors=cols, blurs=blurs)
    t0 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, **kw)
    t1 = codec.decode_tensor(files, None, [(0, 0, 60, 60)] * 3, ops, augments=[None, _Augment(), None], **kw)
    assert torch.equal(t0.view(torch.int16), t1.view(torch.int16))


@gpu
def test_augment_failures(codec):
    """Each refused input fails naming the entry, before anything is written."""
    px, pa = synth.rgb(100, 120, 5), synth.noise(90, 80, 6, channels=4)
    f, fa_ = po.encode(1, px), po.encode(2, pa)
    assert po.decode(fa_).shape[2] == 4

    def call(a1, files=None, fmt=None, boxes=None):
        files = files or [f, f]
        nb = [100 * 120 * 4 * 4] * 2
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, 0xA5, np.uint8)
        err = None
        try:
            codec.decode_augment_raw(fmt, descs, None, None, None if boxes is None else rects(boxes), None, None, None, None,
                                     augment_array([augment_params([("Invert", 0.0)], (1, 1)), a1], 2), 2, fa.ctypes.data, len(fb), 0,
                                     foffs, fsizes, out.ctypes.data, poff, 0)
        except RuntimeError as e:
            err = str(e)
        return err, out

    def prog(**fields):
        a = augment_params([("ShearX", 0.1)], (120, 100))
        for k, v in fields.items():
            if k == "data":
                a.step[0].data[:] = v
            else:
                setattr(a.step[0] if k != "nsteps" else a, k, v)
        return a

    bad = [(prog(nsteps=9), "steps"), (prog(kind=11), "kind"), (prog(arg=1), "resample"), (prog(arg=4), "resample")]
    bad += [(prog(data=[1, 0, math.inf, 0, 1, 0]), "coefficient"), (prog(data=[1, math.nan, 0, 0, 1, 0]), "coefficient"),
            (prog(data=[1, 0, 0, 2.0 ** 64, 1, 0]), "coefficient")]
    bad += [(prog(kind=K["transpose"], arg=7), "op code"), (prog(kind=K["transpose"], arg=-1), "op code"),
            (prog(kind=K["transpose"], arg=0), "quarter")]
    bad += [(prog(kind=K[k], value=v), "factor") for k in ("brightness", "color", "contrast", "sharpness") for v in (-0.1, math.inf, math.nan)]
    bad += [(prog(kind=K["posterize"], arg=9), "bits"), (prog(kind=K["posterize"], arg=-1), "bits"),
            (prog(kind=K["solarize"], value=math.nan), "NaN")]
    for a1, word in bad:
        err, out = call(a1)
        assert err is not None and "entry 1" in err and word in err and (out == 0xA5).all(), (word, err)
    for fmt in (None, tensor_format("float32")):   # any step on an RGBA entry whose output keeps alpha
        err, out = call(augment_params([("Brightness", 0.2)], (1, 1)), [f, fa_], fmt)
        assert err is not None and "entry 1" in err and "alpha" in err and (out == 0xA5).all(), err
    assert call(augment_params([("Equalize", 0.0)], (1, 1)), [f, fa_], tensor_format("float32", drop_alpha=True))[0] is None
    assert call(prog(kind=K["transpose"], arg=0), boxes=[(0, 0, 50, 50)] * 2)[0] is None   # square: a quarter turn is fine
    assert call(augment_params([("Solarize", -math.inf)], (1, 1)))[0] is None
