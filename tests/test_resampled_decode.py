"""Resampled decode (xpngb_decode_resampled / Codec.decode_resized and decode_tensor with filters and windows): entry i is
orient(op, window(resize_f(crop, size))), byte-identical to Pillow's Image.resize(size, f) for its five convolution filters,
and so to torchvision's PIL pipelines such as Resize(256) + CenterCrop(224).

resize_pil() restates Pillow's 8-bit resampling (Resample.c) for every filter in numpy; sin and cos come from Python's
math module, which calls the C library as Pillow does.  It is pinned to the installed Pillow by the CPU tests below.
Without a GPU: resize_pil against PIL, windows of it against torchvision's Resize + CenterCrop, resize_center_crop against
torchvision's size and offset rules, and the accumulator limits.
On the GPU: the device's weight tables against coeffs(), and every output against
po.orient(op, window(resize_pil(po.decode(f)[crop], size, filter)))."""
import ctypes as C
import math

import numpy as np
import pytest
from PIL import Image

from oracle import pyoracle as po
import xpng_b200
from xpng_b200 import synth
from xpng_b200.codec import _Image, filter_codes, op_codes, rects, region_tiles, resize_center_crop, sizes as size_arr, tensor_format
from test_region import GENS, grid_rects, halfflat, scribble_outside
from test_resized_decode import ORACLE_CASES, rrc_boxes

gpu = pytest.mark.gpu
ALL_OPS = list(po.TOOL_OPS)
PREC = 22                                           # Pillow's PRECISION_BITS for 8-bit images
LANCZOS, BILINEAR, BICUBIC, BOX, HAMMING = 1, 2, 3, 4, 5
FILTERS = (LANCZOS, BILINEAR, BICUBIC, BOX, HAMMING)
SUPPORT = {BOX: 0.5, BILINEAR: 1.0, HAMMING: 1.0, BICUBIC: 2.0, LANCZOS: 3.0}
SIDE_MAX = {BOX: 1 << 23, BILINEAR: 1 << 23, HAMMING: 1 << 23, BICUBIC: 1 << 22, LANCZOS: 1 << 21}   # api.cu resize_side_max
NEG_MAX = {BOX: 0.0, BILINEAR: 0.0, HAMMING: 0.0, BICUBIC: 0.25, LANCZOS: 0.375}   # the negative weight sum each limit allows


# ---------------------------------------------------------------------------------------------------- the oracle

_vsin, _vcos = np.frompyfunc(math.sin, 1, 1), np.frompyfunc(math.cos, 1, 1)
HAM_A, HAM_B = float(np.float32(0.54)), float(np.float32(0.46))   # Pillow writes hamming's constants as float literals


def _sinc(x):
    """Pillow's sinc_filter: 1 at 0, else sin(x * pi) / (x * pi)."""
    out = np.ones_like(x)
    nz = x != 0.0
    y = x[nz] * math.pi
    out[nz] = _vsin(y).astype(np.float64) / y
    return out


def filter_values(f, x):
    """Pillow's filter functions (Resample.c) of a float64 array, operation by operation as its C rounds them."""
    out = np.zeros_like(x)
    if f == BOX:
        out[(x > -0.5) & (x <= 0.5)] = 1.0
    elif f == BILINEAR:
        a = np.abs(x)
        out[a < 1.0] = 1.0 - a[a < 1.0]
    elif f == HAMMING:
        a = np.abs(x)
        out[a == 0.0] = 1.0
        m = (a > 0.0) & (a < 1.0)
        y = a[m] * math.pi
        out[m] = _vsin(y).astype(np.float64) / y * (HAM_A + HAM_B * _vcos(y).astype(np.float64))
    elif f == BICUBIC:                                 # a = -0.5
        a = np.abs(x)
        m1, m2 = a < 1.0, (a >= 1.0) & (a < 2.0)
        out[m1] = ((1.5 * a[m1] - 2.5) * a[m1]) * a[m1] + 1.0
        out[m2] = (((a[m2] - 5.0) * a[m2] + 8.0) * a[m2] - 4.0) * -0.5
    elif f == LANCZOS:
        m = (x >= -3.0) & (x < 3.0)
        out[m] = _sinc(x[m]) * _sinc(x[m] / 3.0)
    else:
        raise ValueError(f)
    return out


def coeffs(f, inn, out, first=0, count=None):
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc of one axis for output coordinates first .. first + count - 1:
    xmin, n and (count, ksize) integer weights, zero past each window.  Every float operation is a float64 one, and the
    weight sum is accumulated left to right, as in the C."""
    count = out - first if count is None else count
    scale = inn / out
    fs = max(scale, 1.0)
    support, ss = SUPPORT[f] * fs, 1.0 / fs
    ksize = int(math.ceil(support)) * 2 + 1
    center = (np.arange(first, first + count, dtype=np.float64) + 0.5) * scale
    xmin = np.maximum((center - support + 0.5).astype(np.int64), 0)
    xmax = np.minimum((center + support + 0.5).astype(np.int64), inn)
    n = xmax - xmin
    t = np.arange(ksize)
    valid = t[None, :] < n[:, None]
    x = ((t[None, :] + xmin[:, None]).astype(np.float64) - center[:, None]) + 0.5
    w = np.zeros(x.shape)
    w[valid] = filter_values(f, x[valid] * ss)
    ww = np.cumsum(w, axis=1)[:, -1]                 # sequential: zeros past the window add nothing
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    k = np.trunc(np.where(w < 0.0, -0.5 + w * (1 << PREC), 0.5 + w * (1 << PREC))).astype(np.int64)
    k[~valid] = 0
    return xmin, n, k


def _pass(px, out, axis, f):
    """One resampling pass along axis (0: vertical, 1: horizontal) of an (h, w, c) uint8 array."""
    inn = px.shape[axis]
    if inn == out:
        return px
    xmin, _, k = coeffs(f, inn, out)
    src = np.moveaxis(px.astype(np.int64), axis, 0)
    acc = np.full((out,) + src.shape[1:], 1 << (PREC - 1), np.int64)
    for t in range(k.shape[1]):
        idx = np.minimum(xmin + t, inn - 1)             # weights past the window are 0
        acc += src[idx] * k[:, t].reshape((out,) + (1,) * (src.ndim - 1))
    return np.moveaxis(np.clip(acc >> PREC, 0, 255).astype(np.uint8), 0, axis)


def resize_pil(px, w, h, f):
    """Pillow's Image.resize((w, h), f) of the (h0, w0, c) uint8 array px, every channel on its own: the horizontal pass
    first, rounded to bytes, then the vertical one; vertical first for images more than 100 times taller than wide that
    shrink vertically (Pillow 12)."""
    h0, w0 = px.shape[:2]
    if h < h0 and h0 > 100 * w0:
        return _pass(_pass(px, h, 0, f), w, 1, f)
    return _pass(_pass(px, w, 1, f), h, 0, f)


def window(px, win):
    if win is None:
        return px
    x, y, w, h = win
    return px[y: y + h, x: x + w]


def pil_resize(px, w, h, f):
    return np.asarray(Image.fromarray(px).resize((w, h), f))


def pil_resize_channels(px, w, h, f):
    return np.stack([pil_resize(np.ascontiguousarray(px[:, :, c]), w, h, f) for c in range(px.shape[2])], axis=2)


# ---------------------------------------------------------------------------------------------------- oracle against PIL (CPU)

def resample_cases():
    """The 330 cases of the bilinear tests, plus an identity axis on either side and 1-pixel sides."""
    rng = np.random.default_rng(20261021)
    extra = [((1, 1), (5, 1)), ((1, 9), (1, 3)), ((9, 1), (3, 1)), ((1, 300), (2, 1)), ((300, 1), (1, 2))]
    for _ in range(10):
        h0, w0 = int(rng.integers(1, 300)), int(rng.integers(1, 300))
        extra += [((h0, w0), (w0, int(rng.integers(1, 400)))), ((h0, w0), (int(rng.integers(1, 400)), h0))]
    return list(ORACLE_CASES) + extra


CASES = resample_cases()


def content(k, h0, w0, c):
    """Noise, smooth ramps and checkerboards (the last two drive the negative lobes past 0 and 255)."""
    rng = np.random.default_rng(k)
    px = rng.integers(0, 256, (h0, w0, c), dtype=np.uint8)
    if k % 3 == 1:
        px = np.cumsum(px.astype(np.int64), axis=1).astype(np.uint8)
    elif k % 3 == 2:
        yy, xx = np.mgrid[:h0, :w0]
        px[:] = (((yy // (1 + k % 4) + xx // (1 + k % 5)) % 2) * 255).astype(np.uint8)[:, :, None]
    return px


def test_case_count():
    assert len(CASES) >= 330
    assert sum(1 for (h0, w0), (w, h) in CASES if (w == w0) != (h == h0)) >= 20     # one identity axis
    assert sum(1 for (h0, w0), (w, h) in CASES if h < h0 and h0 > 100 * w0 and w != w0) >= 20   # vertical first
    assert sum(1 for (h0, w0), (w, h) in CASES if w > 2 * w0 and h > 2 * h0) >= 20    # upscales


@pytest.mark.parametrize("f", FILTERS)
@pytest.mark.parametrize("part", range(6))
def test_resample_oracle_matches_pil(f, part):
    for k in range(part, len(CASES), 6):
        (h0, w0), (w, h) = CASES[k]
        px = content(k, h0, w0, 3)
        got = resize_pil(px, w, h, f)
        assert got.shape == (h, w, 3)
        assert np.array_equal(got, pil_resize(px, w, h, f)), (k, f)
        four = np.concatenate([px, content(k + 7, h0, w0, 1)], axis=2)
        assert np.array_equal(resize_pil(four, w, h, f), pil_resize_channels(four, w, h, f)), (k, f)


def test_negative_weights_are_rounded_away_from_zero():
    _, _, k = coeffs(BICUBIC, 5, 17)
    assert (k < 0).any()
    _, _, k = coeffs(LANCZOS, 9, 4)
    assert (k < 0).any()


def _tv_center_crop(pil, resize, crop, mode, max_size=None):
    import torchvision.transforms as T
    return np.asarray(T.Compose([T.Resize(resize, mode, max_size=max_size), T.CenterCrop(crop)])(pil))


@pytest.mark.parametrize("mode", ("bilinear", "bicubic", "lanczos"))
def test_window_is_resize_then_center_crop(mode):
    """window(resize_pil) with resize_center_crop's size and window is torchvision's Resize + CenterCrop of the PIL image:
    landscape and portrait, resized widths 341 and 343 (both parities of the half-pixel offset) and max_size."""
    from torchvision.transforms import InterpolationMode
    im = InterpolationMode(mode)
    f = xpng_b200.codec.filter_code(im)
    cases = [((500, 375), 256, 224, None), ((333, 500), 256, 224, None), ((686, 512), 256, 224, None), ((640, 427), 256, 224, None),
             ((375, 500), 224, 224, None), ((1000, 300), 256, 64, 300), ((300, 1000), 200, (50, 40), 260), ((1920, 1080), 256, 224, None)]
    for k, ((w, h), resize, crop, max_size) in enumerate(cases):
        px = content(k, h, w, 3)
        (W, H), win = resize_center_crop(w, h, resize, crop, max_size)
        got = window(resize_pil(px, W, H, f), win)
        assert np.array_equal(got, _tv_center_crop(Image.fromarray(px), resize, crop, im, max_size)), (w, h, resize, crop)
    assert resize_center_crop(500, 375, 256, 224)[0] == (341, 256) and resize_center_crop(686, 512, 256, 224)[0] == (343, 256)
    assert resize_center_crop(500, 375, 256, 224)[1][:2] == (58, 16)      # round(58.5) == 58: half to even


def test_resize_center_crop_matches_torchvision_rules():
    import torch
    import torchvision.transforms.functional as F
    rng = np.random.default_rng(5)
    for _ in range(400):
        w, h = int(rng.integers(1, 3000)), int(rng.integers(1, 3000))
        if rng.integers(2):
            resize, max_size = int(rng.integers(1, 400)), None
            if rng.integers(2):
                max_size = resize + int(rng.integers(1, 500))
        else:
            resize, max_size = (int(rng.integers(1, 400)), int(rng.integers(1, 400))), None
        H, W = F._compute_resized_output_size((h, w), [resize] if isinstance(resize, int) else list(resize), max_size)
        crop = (int(rng.integers(1, H + 3)), int(rng.integers(1, W + 3)))
        if crop[0] > H or crop[1] > W:
            with pytest.raises(ValueError):
                resize_center_crop(w, h, resize, crop, max_size)
            continue
        size, win = resize_center_crop(w, h, resize, crop, max_size)
        idx = torch.arange(H * W).reshape(1, H, W)
        c = F.center_crop(idx, list(crop))
        top, left = divmod(int(c[0, 0, 0]), W)
        assert size == (W, H) and win == (left, top, crop[1], crop[0]), (w, h, resize, crop, max_size)


def _neg_mass(f, inn, out):
    """The largest sum of negative normalised weights of any output coordinate of an inn -> out axis."""
    xmin, n, k = coeffs(f, inn, out)
    return float(np.where(k < 0, -k, 0).sum(axis=1).max()) / (1 << PREC)


def test_accumulator_limits():
    """At each filter's crop-side limit L (n <= L taps), the widest partial sum, 2^21 + 255 * (2^22 * (1 + 2N) + L / 2),
    fits in int32 for the negative weight sum N it allows; the sums N measured here stay below that allowance, including
    the largest ones found over every in, out <= 256 (bicubic 208 -> 193, lanczos 4 -> 5)."""
    for f in FILTERS:
        worst = (1 << 21) + 255 * ((1 << PREC) * (1 + 2 * NEG_MAX[f]) + SIDE_MAX[f] / 2)
        assert worst < 2 ** 31, f
    sweep = {f: max(_neg_mass(f, i, o) for i in range(1, 49) for o in range(1, 49) if i != o) for f in FILTERS}
    assert sweep[BOX] == sweep[BILINEAR] == sweep[HAMMING] == 0.0
    for f, (i, o), n in ((BICUBIC, (208, 193), 0.1344), (LANCZOS, (4, 5), 0.2858)):
        assert abs(_neg_mass(f, i, o) - n) < 1e-3
        assert max(sweep[f], n) < NEG_MAX[f]


def test_filter_names():
    from torchvision.transforms import InterpolationMode
    assert list(filter_codes([Image.Resampling.BICUBIC, "lanczos", InterpolationMode.BOX, 5, "Bilinear"], 5)) == [3, 1, 4, 5, 2]
    assert list(filter_codes("hamming", 3)) == [5, 5, 5]
    for bad in (0, Image.Resampling.NEAREST, InterpolationMode.NEAREST, "nearest", 6, "cubic"):
        with pytest.raises(ValueError):
            filter_codes(bad, 1)


# ---------------------------------------------------------------------------------------------------- resampled decode (GPU)

@pytest.fixture(scope="module")
def codec():
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


@gpu
def test_weight_tables_match_host_libm(codec):
    """The device's tables (CUDA's sin and cos for hamming and lanczos) against coeffs() (the C library's, as Pillow), for
    every in in 1..1024 against seeded up- and downscales, and at offsets first > 0."""
    rng = np.random.default_rng(1024)
    pairs, bad = 0, []
    for inn in range(1, 1025):
        outs = {inn + int(rng.integers(1, 400)), int(rng.integers(1, 5)), max(1, inn // int(rng.integers(2, 9))), int(rng.integers(1, 2 * inn + 2))}
        for out in sorted(outs - {inn}):
            first = int(rng.integers(0, out)) if out > 1 and inn % 3 == 0 else 0
            for f in FILTERS:
                xn, k = codec.resize_coeffs(f, inn, out, first)
                xmin, n, kw = coeffs(f, inn, out, first)
                pairs += 1
                if not (np.array_equal(xn[:, 0], xmin) and np.array_equal(xn[:, 1], n) and np.array_equal(k, kw)):
                    bad.append((f, inn, out, first))
    print(f"weight tables: {pairs} (filter, in, out) tables, {len(bad)} mismatches")
    assert pairs > 15000 and not bad, bad[:20]


def want_of(full, size, f, op=None, rect=None, win=None):
    crop = full if rect is None else window(full, rect)
    return po.orient(op or "tl", window(resize_pil(crop, size[0], size[1], f), win))


def check(codec, files, szs, boxes, ops, filters, wins):
    got = codec.decode_resized(files, szs, boxes, ops, filters, wins)
    fulls = {}
    for i, (f, z, g) in enumerate(zip(files, szs, got)):
        if f not in fulls:
            fulls[f] = po.decode(f)
        want = want_of(fulls[f], z, filters if not isinstance(filters, list) else filters[i], None if ops is None else ops[i],
                       None if boxes is None else boxes[i], None if wins is None else wins[i])
        assert g.shape == want.shape and np.array_equal(g, want), (i, z, boxes and boxes[i], ops and ops[i], wins and wins[i])
    return got


def window_kinds(W, H, rng):
    """The whole image, the four corners, 1 x 1 at a corner, full-height and full-width strips at the edges, an interior
    window and the center crop."""
    cw, ch = max(1, W // 3), max(1, H // 3)
    return [(0, 0, W, H), (0, 0, cw, ch), (W - cw, 0, cw, ch), (0, H - ch, cw, ch), (W - cw, H - ch, cw, ch),
            (W - 1, H - 1, 1, 1), (0, 0, 1, 1), (0, 0, cw, H), (W - cw, 0, cw, H), (0, H - ch, W, ch),
            (int(rng.integers(W)) // 2, int(rng.integers(H)) // 2, cw, ch), (int(round((W - cw) / 2.0)), int(round((H - ch) / 2.0)), cw, ch)]


def size_kinds(w, h):
    return [(224, 224), (max(1, int(w * 1.7)), max(1, int(h * 1.7))), (max(1, w // 3), h * 2), (w, max(1, h // 4)), (1, 1), (w, h)]


@gpu
@pytest.mark.parametrize("level", (1, 2, 7))
@pytest.mark.parametrize("gen", sorted(GENS))
def test_resampled_against_oracle(codec, gen, level):
    rng = np.random.default_rng(sorted(GENS).index(gen) * 3 + level + 300)
    h, w = 700, 1000
    f = po.encode(level, GENS[gen](h, w, 46))
    files, szs, boxes, ops, filters, wins = [], [], [], [], [], []
    for j, r in enumerate(grid_rects(w, h, rng)):
        for m, z in enumerate(size_kinds(r[2], r[3])):
            kinds = window_kinds(*z, rng)
            files.append(f); szs.append(z); boxes.append(r)
            ops.append(ALL_OPS[(j + m) % len(ALL_OPS)]); filters.append(FILTERS[(3 * j + m) % len(FILTERS)])
            wins.append(kinds[(5 * j + m) % len(kinds)])
    check(codec, files, szs, boxes, ops, filters, wins)
    for fl in FILTERS:                                       # whole images, every window kind, one filter per call
        kinds = window_kinds(300, 200, rng)
        check(codec, [f] * len(kinds), [(300, 200)] * len(kinds), None, None, fl, kinds)


@gpu
def test_resampled_mixed_batch(codec):
    """Every filter and window kind in one call, with identity axes, vertical-first crops and the stored level."""
    imgs = [synth.rgb(900, 1300, 1), synth.rgba(500, 460, 2), synth.gray_as_rgb(300, 520, 3), synth.noise(90, 70, 4),
            np.full((700, 800, 3), 9, np.uint8), synth.rgb(1, 1399, 6), synth.rgb(1823, 1, 5), synth.rgba(333, 129, 7)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7, 1, 2, 2, 1, 7), imgs)]
    rng = np.random.default_rng(13)
    batch, boxes, szs, ops, filters, wins = [], [], [], [], [], []
    for f, im in zip(files, imgs):
        h, w = im.shape[:2]
        for k in range(6):
            x0, y0 = int(rng.integers(w)), int(rng.integers(h))
            r = (0, 0, w, h) if k == 0 else (x0, y0, int(rng.integers(1, w - x0 + 1)), int(rng.integers(1, h - y0 + 1)))
            z = (int(rng.integers(1, 400)), int(rng.integers(1, 400))) if k < 3 else (r[2], int(rng.integers(1, 300))) if k == 3 else \
                (int(rng.integers(1, 300)), r[3]) if k == 4 else (r[2], r[3])
            kinds = window_kinds(*z, rng)
            batch.append(f); boxes.append(r); szs.append(z)
            ops.append(ALL_OPS[int(rng.integers(len(ALL_OPS)))]); filters.append(FILTERS[int(rng.integers(5))])
            wins.append(kinds[int(rng.integers(len(kinds)))])
    for f, r, z in ((files[0], (5, 0, 8, 900), (224, 224)), (files[6], (0, 0, 1, 1823), (3, 500)), (files[2], (7, 0, 2, 300), (9, 5))):
        for fl in (LANCZOS, BICUBIC):
            batch.append(f); boxes.append(r); szs.append(z); ops.append("r90"); filters.append(fl)
            wins.append((0, z[1] // 3, z[0], max(1, z[1] // 2)))
    perm = rng.permutation(len(batch))
    pick = lambda a: [a[k] for k in perm]
    check(codec, pick(batch), pick(szs), pick(boxes), pick(ops), pick(filters), pick(wins))


@gpu
def test_defaults_are_resized_and_tensor_decode(codec):
    """filters == NULL and windows == NULL through the new entry point, and all-bilinear filters with whole windows, give
    the bytes of xpngb_decode_resized and xpngb_decode_tensor."""
    import torch
    imgs = [synth.rgb(700, 1000, 11), synth.rgba(500, 460, 12), synth.rgb(1823, 3, 13), synth.rgb(333, 517, 14)]
    files = [po.encode(lv, im) for lv, im in zip((1, 2, 7, 1), imgs)]
    boxes = [(10, 20, 600, 400), (0, 0, 460, 500), (0, 0, 3, 1823), (5, 5, 500, 300)]
    szs = [(224, 224), (100, 333), (2, 50), (500, 300)]
    ops = ["r90", "mh", "tl", "mvh"]
    want = codec.decode_resized(files, szs, boxes, ops)
    for filters, wins in ((None, None), ("bilinear", None), (None, [(0, 0, w, h) for w, h in szs]), ([2] * 4, [(0, 0, w, h) for w, h in szs])):
        nb = [w * h * im.shape[2] for (w, h), im in zip(szs, imgs)]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.zeros(poff + 16, np.uint8)
        codec.decode_resampled_raw(None, descs, filter_codes(filters, 4), op_codes(ops), rects(boxes), size_arr(szs),
                                   None if wins is None else rects(wins), 4, fa.ctypes.data, len(fb), 0, foffs, fsizes,
                                   out.ctypes.data, poff, 0)
        for i, g in enumerate(want):
            assert out[descs[i].offset: descs[i].offset + g.size].tobytes() == g.tobytes(), (filters, wins, i)
    f3 = [files[0], files[3]]
    t0 = codec.decode_tensor(f3, [(224, 224)] * 2, [boxes[0], boxes[3]], ["mh", "tl"], torch.bfloat16, mean=(0.5, 0.4, 0.3), std=(0.2, 0.3, 0.4))
    t1 = codec.decode_tensor(f3, [(224, 224)] * 2, [boxes[0], boxes[3]], ["mh", "tl"], torch.bfloat16, mean=(0.5, 0.4, 0.3), std=(0.2, 0.3, 0.4),
                             filters="bilinear", windows=[(0, 0, 224, 224)] * 2)
    assert torch.equal(t0.view(torch.int16), t1.view(torch.int16))


@gpu
def test_only_the_support_is_decoded(codec):
    """Tiles outside the cover of a window's support (widened by one pixel, as the library decodes it) are scribbled over;
    the call still returns the right pixels."""
    rng = np.random.default_rng(77)
    for level in (1, 2):
        h, w = 1400, 2000
        px = synth.rgb(h, w, 90 + level)
        f = po.encode(level, px)
        for crop, z, win, fl in (((0, 0, w, h), (500, 350), (400, 250, 100, 100), LANCZOS),
                                 ((100, 50, 1800, 1300), (224, 224), (0, 0, 50, 224), BICUBIC),
                                 ((0, 0, w, h), (4000, 2800), (3000, 100, 64, 64), HAMMING),
                                 ((0, 0, w, h), (w, 300), (1500, 10, 400, 20), BOX)):
            span = []
            for axis, (c0, cn, zn, w0, wn) in enumerate(((crop[0], crop[2], z[0], win[0], win[2]), (crop[1], crop[3], z[1], win[1], win[3]))):
                if cn == zn:
                    span.append((c0 + w0, wn))
                    continue
                xmin, n, _ = coeffs(fl, cn, zn, w0, wn)
                lo, hi = max(int(xmin[0]) - 1, 0), min(int(xmin[-1] + n[-1]) + 1, cn)
                span.append((c0 + lo, hi - lo))
            _, cover = region_tiles(w, h, (span[0][0], span[1][0], span[0][1], span[1][1]))
            g = scribble_outside(f, w, h, cover, int(rng.integers(1 << 30)))
            got = codec.decode_resized([g], [z], [crop], None, fl, [win])[0]
            assert np.array_equal(got, want_of(px, z, fl, None, crop, win)), (level, crop, z, win)


def pack(files, out_sizes):
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
def test_resampled_pipelined_chunks_device_resident(monkeypatch):
    """Sintel-like frames, one RandomResizedCrop box each, every filter and a window per entry, cut into several chunks on
    three lanes, with files and output in device memory."""
    import torch
    frames = synth.sintel_batch(range(1000, 1024))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "1")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "3")
    monkeypatch.setenv("XPNGB_CHUNK_MPIX", "3")
    cd = xpng_b200.Codec(0)
    try:
        rng = np.random.default_rng(67)
        n = len(frames)
        boxes = rrc_boxes(rng, n)
        ops = [ALL_OPS[int(rng.integers(len(ALL_OPS)))] for _ in frames]
        filters = [FILTERS[k % 5] for k in range(n)]
        szs = [(224, 224) if k % 2 else (256, 256 + k) for k in range(n)]
        wins = [window_kinds(*z, rng)[k % 12] for k, z in enumerate(szs)]
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            nb = [ww * wh * 3 for (_, _, ww, wh) in wins]
            descs, foffs, fsizes, fb, poff = pack(files, nb)
            dfiles = torch.from_numpy(np.frombuffer(fb, np.uint8).copy()).cuda()
            dpx = torch.zeros(poff, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            cd.decode_resampled_raw(None, descs, filter_codes(filters, n), op_codes(ops), rects(boxes), size_arr(szs), rects(wins), n,
                                    dfiles.data_ptr(), len(fb), 1, foffs, fsizes, dpx.data_ptr(), poff, 1)
            out = dpx.cpu().numpy()
            for i in range(n):
                want = want_of(frames[i], szs[i], filters[i], ops[i], boxes[i], wins[i])
                got = out[descs[i].offset: descs[i].offset + want.size].reshape(want.shape)
                assert np.array_equal(got, want), (lv, i)
            assert cd.decode_resized(files[:8], szs[:8], boxes[:8], ops[:8], filters[:8], wins[:8])[3].shape == \
                want_of(frames[3], szs[3], filters[3], ops[3], boxes[3], wins[3]).shape
    finally:
        cd.close()


# ---------------------------------------------------------------------------------------------------- torchvision pipelines (GPU)

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
CLIP = ((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711))
ASPECTS = [(500, 375), (333, 500), (640, 427), (427, 640), (686, 512), (300, 300), (1024, 683), (375, 500)]


def _eval_batch(level):
    imgs = [synth.rgb(h, w, 500 + k) for k, (w, h) in enumerate(ASPECTS)]
    return imgs, [po.encode(level, im) for im in imgs]


@gpu
@pytest.mark.parametrize("level", (1, 2))
def test_torchvision_eval_pipelines(codec, level):
    """One decode_tensor call per batch against torch.stack of the transforms on PIL images, bit for bit: ImageNet's
    Resize(256, BICUBIC) + CenterCrop(224) in v1 and v2, float32 and bfloat16, and CLIP's Resize(224) + CenterCrop(224)."""
    import torch
    import torchvision.transforms as T
    import torchvision.transforms.v2 as v2
    B = T.InterpolationMode.BICUBIC
    imgs, files = _eval_batch(level)
    pils = [Image.fromarray(im) for im in imgs]
    for resize, (mean, std) in ((256, IMAGENET), (224, CLIP)):
        geo = [resize_center_crop(im.shape[1], im.shape[0], resize, 224) for im in imgs]
        assert len({z for z, _ in geo}) > 1                     # ragged before the window
        szs, wins = [z for z, _ in geo], [w for _, w in geo]
        for dtype in (torch.float32, torch.bfloat16):
            v1 = T.Compose([T.Resize(resize, B), T.CenterCrop(224), T.ToTensor(), T.Normalize(mean, std)])
            want = torch.stack([v1(p) for p in pils]).to(dtype)
            got = codec.decode_tensor(files, szs, None, None, dtype, mean=mean, std=std, filters=B, windows=wins).cpu()
            assert got.shape == want.shape and torch.equal(got.view(torch.int16 if dtype == torch.bfloat16 else torch.int32),
                                                           want.view(torch.int16 if dtype == torch.bfloat16 else torch.int32)), (resize, dtype)
            tv2 = v2.Compose([v2.Resize(resize, B), v2.CenterCrop(224), v2.ToImage(), v2.ToDtype(torch.float32, scale=True), v2.Normalize(mean, std)])
            want = torch.stack([tv2(p) for p in pils]).to(dtype)
            got = codec.decode_tensor(files, szs, None, None, dtype, scale="mul", mean=mean, std=std, filters=B, windows=wins).cpu()
            assert torch.equal(got.view(torch.int16 if dtype == torch.bfloat16 else torch.int32),
                               want.view(torch.int16 if dtype == torch.bfloat16 else torch.int32)), (resize, dtype, "v2")


@gpu
def test_torchvision_random_resized_crop(codec):
    """RandomResizedCrop(224, BICUBIC) + RandomHorizontalFlip through sizes, rects and ops."""
    import torch
    import torchvision.transforms as T
    import torchvision.transforms.functional as F
    imgs, files = _eval_batch(2)
    torch.manual_seed(3)
    boxes, ops, want = [], [], []
    for im in imgs:
        p = Image.fromarray(im)
        i, j, h, w = T.RandomResizedCrop.get_params(p, (0.08, 1.0), (3 / 4, 4 / 3))
        flip = bool(torch.rand(1) < 0.5)
        r = F.resized_crop(p, i, j, h, w, [224, 224], T.InterpolationMode.BICUBIC)
        if flip:
            r = F.hflip(r)
        want.append(F.normalize(F.to_tensor(r), *IMAGENET))
        boxes.append((j, i, w, h)); ops.append("mh" if flip else "tl")
    got = codec.decode_tensor(files, [(224, 224)] * len(files), boxes, ops, torch.float32, mean=IMAGENET[0], std=IMAGENET[1],
                              filters="bicubic").cpu()
    assert torch.equal(got.view(torch.int32), torch.stack(want).view(torch.int32))


# ---------------------------------------------------------------------------------------------------- failures (GPU)

@gpu
def test_resampled_failures(codec):
    px = synth.rgb(600, 700, 5)
    f = po.encode(1, px)

    def call(files, szs, filters=None, wins=None, cap_delta=0, fmt=None):
        nb = [ww * wh * 3 if 0 < ww <= 1 << 24 and 0 < wh <= 1 << 24 else 16 for (ww, wh) in
              ([(w_[2], w_[3]) for w_ in wins] if wins is not None else szs)]
        if fmt is not None:
            nb = [4 * b for b in nb]
        descs, foffs, fsizes, fb, poff = pack(files, nb)
        fa = np.frombuffer(fb, np.uint8)
        out = np.full(poff + 64, 0xA5, np.uint8)
        err = None
        try:
            codec.decode_resampled_raw(fmt, descs, None if filters is None else (C.c_int * len(filters))(*filters), None, None,
                                       size_arr(szs), None if wins is None else rects(wins), len(files), fa.ctypes.data, len(fb), 0,
                                       foffs, fsizes, out.ctypes.data, poff + cap_delta, 0)
        except RuntimeError as e:
            err = str(e)
        return err, out

    for bad in (0, 6, -1):
        err, out = call([f, f], [(10, 10), (224, 224)], filters=[3, bad])
        assert err is not None and "entry 1" in err and "filter" in err and (out == 0xA5).all(), (bad, err)
    for win in ((0, 0, 0, 5), (0, 0, 5, 0), (220, 0, 5, 5), (0, 224, 1, 1), (2 ** 63, 0, 1, 1), (0, 0, 225, 224)):
        err, out = call([f, f], [(10, 10), (224, 224)], wins=[(0, 0, 10, 10), win])
        assert err is not None and "entry 1" in err and "window" in err and (out == 0xA5).all(), (win, err)
    err, out = call([f], [(224, 224)], wins=[(10, 10, 100, 100)], cap_delta=-1)     # past out_cap (the window, not the size)
    assert "exceed" in err and (out == 0xA5).all()
    err, out = call([f], [(224, 224)], wins=[(10, 10, 100, 100)], cap_delta=-1, fmt=tensor_format("float32"))
    assert "exceed" in err and (out == 0xA5).all()
    assert call([f], [(224, 224)], wins=[(10, 10, 100, 100)])[0] is None
    # a crop side past the filter's accumulator limit (a stored single-row image: no tiles to decode)
    wide = po.encode(7, np.zeros((1, (1 << 21) + 1, 3), np.uint8))
    err, out = call([f, wide], [(10, 10), (1, 1)], filters=[2, LANCZOS])
    assert err is not None and "entry 1" in err and "crop side" in err and (out == 0xA5).all(), err
    descs, foffs, fsizes, fb, poff = pack([f], [224 * 224 * 3])
    fa = np.frombuffer(fb, np.uint8)
    out = np.full(poff + 16, 0xA5, np.uint8)
    assert xpng_b200.lib().xpngb_decode_resampled(codec._h, None, None, None, descs, None, None, None, 1, fa.ctypes.data, len(fb), 0,
                                                  foffs, fsizes, out.ctypes.data, poff, 0) != 0
    assert "sizes" in codec._err() and (out == 0xA5).all()
    with pytest.raises(RuntimeError, match="entry 1"):
        codec.decode_resized([f, f], [(5, 5), (9, 9)], filters=[2, 0 + 3], windows=[(0, 0, 5, 5), (8, 8, 2, 1)])
    with pytest.raises(ValueError):
        codec.decode_resized([f], [(5, 5)], filters="nearest")
    # and the context still decodes afterwards
    assert np.array_equal(codec.decode_resized([f], [(224, 224)], None, ["mh"], "lanczos", [(3, 4, 100, 50)])[0],
                          want_of(px, (224, 224), LANCZOS, "mh", None, (3, 4, 100, 50)))
