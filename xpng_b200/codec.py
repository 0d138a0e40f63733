"""ctypes mirror of include/xpng_b200.h (batch C ABI) and include/xpng.h / seven.h (file API).

Names and argument meaning follow the reference: `xpng_store(mode, pm, path)`, `xpng_load(path)`,
`load_7`, `store_7` (xpng.h:12-20, 7/seven.h:3-4); errors are the reference's "returns 1", surfaced
here as exceptions carrying xpngb_last_error().
"""
import ctypes as C
import math
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


class LibraryMissing(RuntimeError):
    pass


def lib_path():
    # XPNGB_LIB: developer override for A/B builds of the same library (tools/abtest.sh)
    return os.environ.get("XPNGB_LIB") or os.path.join(HERE, "libxpng_b200.so")


class _Image(C.Structure):
    _fields_ = [("w", C.c_uint64), ("h", C.c_uint64), ("offset", C.c_uint64), ("A", C.c_uint32), ("mode", C.c_uint32)]


class _Rect(C.Structure):  # xpngb_rect: pixels, (x, y) = top-left corner
    _fields_ = [("x", C.c_uint64), ("y", C.c_uint64), ("w", C.c_uint64), ("h", C.c_uint64)]


class _Size(C.Structure):  # xpngb_size: output pixels of a resized decode
    _fields_ = [("w", C.c_uint32), ("h", C.c_uint32)]


class _Tensor(C.Structure):  # xpngb_tensor: the format of a tensor decode (see tensor_format)
    _fields_ = [("dtype", C.c_uint32), ("layout", C.c_uint32), ("scale", C.c_uint32), ("channels", C.c_uint32),
                ("mean", C.c_float * 4), ("std", C.c_float * 4)]


class _Color(C.Structure):  # xpngb_color: one entry's ColorJitter / RandomGrayscale (see color_params)
    _fields_ = [("order", C.c_uint8 * 4), ("on", C.c_uint32), ("gray", C.c_uint32), ("factor", C.c_double * 4)]


class _Blur(C.Structure):  # xpngb_blur: one entry's GaussianBlur / solarize (see blur_params)
    _fields_ = [("radius", C.c_double * 2), ("solarize", C.c_uint32), ("threshold", C.c_double)]


class _AugStep(C.Structure):  # xpngb_aug_step: one step of an entry's augment program (see augment_params)
    _fields_ = [("data", C.c_double * 6), ("value", C.c_double), ("kind", C.c_uint32), ("arg", C.c_int32), ("fill", C.c_uint8 * 4)]


AUG_STEPS_MAX = 8   # XPNGB_AUG_STEPS_MAX


class _Augment(C.Structure):  # xpngb_augment: one entry's AutoAugment / RandAugment / TrivialAugmentWide ops
    _fields_ = [("nsteps", C.c_uint32), ("step", _AugStep * AUG_STEPS_MAX)]


class _Xpng(C.Structure):  # xpng_t, xpng.h:10
    _fields_ = [("p", C.c_void_p), ("w", C.c_uint64), ("h", C.c_uint64), ("s", C.c_uint64), ("A", C.c_bool)]


_lib = None


def lib():
    """Load libxpng_b200.so; there is no fallback when it is absent."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise LibraryMissing(f"{p} not built: run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C xpng_b200`")
        L = C.CDLL(p)
        vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
        L.xpngb_create.restype = C.c_int; L.xpngb_create.argtypes = [C.POINTER(vp), C.c_int]
        L.xpngb_destroy.restype = None; L.xpngb_destroy.argtypes = [vp]
        L.xpngb_last_error.restype = C.c_char_p; L.xpngb_last_error.argtypes = [vp]
        L.xpngb_encode_bound.restype = u64; L.xpngb_encode_bound.argtypes = [C.POINTER(_Image), u32]
        L.xpngb_encode.restype = C.c_int
        L.xpngb_encode.argtypes = [vp, C.c_int, C.POINTER(_Image), u32, vp, u64, C.c_int, vp, u64, C.c_int,
                                   C.POINTER(u64), C.POINTER(u64)]
        L.xpngb_transform.restype = C.c_int
        L.xpngb_transform.argtypes = [vp, C.c_int, C.POINTER(_Image), u32, vp, u64, C.c_int, vp, C.c_int]
        L.xpngb_encode_oriented.restype = C.c_int
        L.xpngb_encode_oriented.argtypes = [vp, C.c_int, C.c_int, C.POINTER(_Image), u32, vp, u64, C.c_int, vp, u64, C.c_int,
                                            C.POINTER(u64), C.POINTER(u64)]
        L.xpngb_peek.restype = C.c_int; L.xpngb_peek.argtypes = [vp, u64, C.POINTER(_Image)]
        L.xpngb_decode.restype = C.c_int
        L.xpngb_decode.argtypes = [vp, C.POINTER(_Image), u32, vp, u64, C.c_int, C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_region_tiles.restype = u32; L.xpngb_region_tiles.argtypes = [u64, u64, C.POINTER(_Rect), C.POINTER(_Rect)]
        L.xpngb_decode_region.restype = C.c_int
        L.xpngb_decode_region.argtypes = [vp, C.POINTER(_Image), C.POINTER(_Rect), u32, vp, u64, C.c_int, C.POINTER(u64), C.POINTER(u64),
                                          vp, u64, C.c_int]
        L.xpngb_decode_oriented.restype = C.c_int
        L.xpngb_decode_oriented.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(_Image), C.POINTER(_Rect), u32, vp, u64, C.c_int,
                                            C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_resized.restype = C.c_int
        L.xpngb_decode_resized.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(_Image), C.POINTER(_Rect), C.POINTER(_Size), u32, vp, u64,
                                           C.c_int, C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_tensor.restype = C.c_int
        L.xpngb_decode_tensor.argtypes = [vp, C.POINTER(_Tensor), C.POINTER(C.c_int), C.POINTER(_Image), C.POINTER(_Rect), C.POINTER(_Size),
                                          u32, vp, u64, C.c_int, C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_resampled.restype = C.c_int
        L.xpngb_decode_resampled.argtypes = [vp, C.POINTER(_Tensor), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_Image),
                                             C.POINTER(_Rect), C.POINTER(_Size), C.POINTER(_Rect), u32, vp, u64, C.c_int, C.POINTER(u64),
                                             C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_color.restype = C.c_int
        L.xpngb_decode_color.argtypes = [vp, C.POINTER(_Tensor), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_Image), C.POINTER(_Rect),
                                         C.POINTER(_Size), C.POINTER(_Rect), C.POINTER(_Color), u32, vp, u64, C.c_int, C.POINTER(u64),
                                         C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_blur.restype = C.c_int
        L.xpngb_decode_blur.argtypes = [vp, C.POINTER(_Tensor), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_Image), C.POINTER(_Rect),
                                        C.POINTER(_Size), C.POINTER(_Rect), C.POINTER(_Color), C.POINTER(_Blur), u32, vp, u64, C.c_int,
                                        C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_decode_augment.restype = C.c_int
        L.xpngb_decode_augment.argtypes = [vp, C.POINTER(_Tensor), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_Image),
                                           C.POINTER(_Rect), C.POINTER(_Size), C.POINTER(_Rect), C.POINTER(_Color), C.POINTER(_Blur),
                                           C.POINTER(_Augment), u32, vp, u64, C.c_int, C.POINTER(u64), C.POINTER(u64), vp, u64, C.c_int]
        L.xpngb_blur_box.restype = C.c_int
        L.xpngb_blur_box.argtypes = [C.c_double, C.POINTER(C.c_int32), C.POINTER(u32), C.POINTER(u32)]
        L.xpngb_resize_ksize.restype = u32; L.xpngb_resize_ksize.argtypes = [C.c_int, u32, u32]
        L.xpngb_resize_coeffs.restype = C.c_int
        L.xpngb_resize_coeffs.argtypes = [vp, C.c_int, u32, u32, u32, u32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.xpngb_last_kernel_ms.restype = C.c_float; L.xpngb_last_kernel_ms.argtypes = [vp]
        L.xpngb_last_launches.restype = u32; L.xpngb_last_launches.argtypes = [vp]
        L.xpngb_last_tiles.restype = u64; L.xpngb_last_tiles.argtypes = [vp]
        L.xpngb_stream.restype = vp; L.xpngb_stream.argtypes = [vp]
        L.xpngb_profile.restype = None; L.xpngb_profile.argtypes = [vp, C.c_int]
        L.xpngb_profile_report.restype = u32; L.xpngb_profile_report.argtypes = [vp, C.c_char_p, u32]
        L.xpngb_ycocg_forward.restype = C.c_int; L.xpngb_ycocg_forward.argtypes = [vp, vp, vp, u64]
        L.xpngb_ycocg_inverse.restype = C.c_int; L.xpngb_ycocg_inverse.argtypes = [vp, vp, vp, u64]
        # frame batches sharded over devices / ranks (host C, no NCCL): include/xpng_b200.h
        L.xpngb_shard_range.restype = None; L.xpngb_shard_range.argtypes = [u32, u32, u32, C.POINTER(u32), C.POINTER(u32)]
        L.xpngb_packed_offsets.restype = None
        L.xpngb_packed_offsets.argtypes = [C.POINTER(u64), u32, C.POINTER(u64), C.POINTER(u64)]
        L.xpngb_pool_create.restype = C.c_int; L.xpngb_pool_create.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), u32]
        L.xpngb_pool_destroy.restype = None; L.xpngb_pool_destroy.argtypes = [vp]
        L.xpngb_pool_size.restype = u32; L.xpngb_pool_size.argtypes = [vp]
        L.xpngb_pool_last_error.restype = C.c_char_p; L.xpngb_pool_last_error.argtypes = [vp]
        L.xpngb_pool_encode.restype = C.c_int
        L.xpngb_pool_encode.argtypes = [vp, C.c_int, C.POINTER(_Image), u32, vp, u64, vp, u64, C.POINTER(u64), C.POINTER(u64)]
        L.xpngb_pool_decode.restype = C.c_int
        L.xpngb_pool_decode.argtypes = [vp, C.POINTER(_Image), u32, vp, u64, C.POINTER(u64), C.POINTER(u64), vp, u64]
        L.xpngb_gather_open.restype = C.c_int; L.xpngb_gather_open.argtypes = [C.POINTER(vp), C.c_char_p, u32, u32, u32]
        L.xpngb_gather_sizes.restype = C.c_int
        L.xpngb_gather_sizes.argtypes = [vp, u32, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
        L.xpngb_gather_close.restype = None; L.xpngb_gather_close.argtypes = [vp]
        for name in ("xpng_store", "xpng_load", "xpng_from_jpg", "xpng_store_T", "xpng_load_T", "xpng_from_jpg_T", "store_7", "load_7"):
            getattr(L, name).restype = C.c_bool
        L.xpng_store.argtypes = [u64, C.POINTER(_Xpng), C.c_char_p]
        L.xpng_store_T.argtypes = [u64, u64, C.POINTER(_Xpng), C.c_char_p]
        L.xpng_load.argtypes = [C.c_char_p, C.POINTER(_Xpng)]
        L.xpng_load_T.argtypes = [u64, C.c_char_p, C.POINTER(_Xpng)]
        L.xpng_from_jpg.argtypes = [C.c_char_p, C.c_char_p]
        L.store_7.argtypes = [C.POINTER(_Xpng), C.c_char_p]
        L.load_7.argtypes = [C.c_char_p, C.POINTER(_Xpng)]
        _lib = L
    return _lib


OPS = {"r90": 0, "r270": 1, "mv": 2, "mh": 3, "mvh": 4, "tl": 5, "tr": 6}   # include/xpng_b200.h, order of tool.c:133
QUARTER_TURNS = ("r90", "r270")


def inverse_op(name):
    """The op that undoes `name`: decoding a file written by encode_oriented(level, name, ...) with it gives the original
    orientation back.  r90 and r270 undo each other; every other op undoes itself."""
    if name not in OPS:
        raise ValueError(f"unknown op {name!r}")
    return {"r90": "r270", "r270": "r90"}.get(name, name)


def op_codes(names):
    """[op name] -> ctypes array of XPNGB_OP_* codes."""
    bad = [o for o in names if o not in OPS]
    if bad:
        raise ValueError(f"unknown op {bad[0]!r}")
    return (C.c_int * len(names))(*(OPS[o] for o in names))


def _align16(v):
    return (v + 15) & ~15


def rects(boxes):
    """[(x, y, w, h)] -> ctypes array of xpngb_rect."""
    arr = (_Rect * len(boxes))()
    for i, (x, y, w, h) in enumerate(boxes):
        arr[i].x, arr[i].y, arr[i].w, arr[i].h = int(x), int(y), int(w), int(h)
    return arr


def sizes(whs):
    """[(w, h)] -> ctypes array of xpngb_size."""
    arr = (_Size * len(whs))()
    for i, (w, h) in enumerate(whs):
        arr[i].w, arr[i].h = int(w), int(h)
    return arr


_sizes = sizes   # Codec.decode_resized's argument of the same name hides it

FILTERS = {"lanczos": 1, "bilinear": 2, "bicubic": 3, "box": 4, "hamming": 5}   # XPNGB_LANCZOS .. = PIL.Image.Resampling


def filter_code(f):
    """A resampling filter as Pillow numbers it: a name ("bicubic"), a PIL.Image.Resampling value or a torchvision
    InterpolationMode (whose .value is the name).  NEAREST is refused: Pillow does not resize with it by convolution."""
    if not isinstance(f, int):
        name = getattr(f, "value", f)
        if isinstance(name, str) and name.lower() in FILTERS:
            return FILTERS[name.lower()]
        raise ValueError(f"unknown resampling filter {f!r}: one of {sorted(FILTERS)}")
    if int(f) not in FILTERS.values():
        raise ValueError(f"unknown resampling filter {f!r}: one of {sorted(FILTERS)} (PIL.Image.Resampling numbers)")
    return int(f)


def filter_codes(filters, n):
    """None, one filter for all n entries, or a list of n -> ctypes array of filter codes (None for None)."""
    if filters is None:
        return None
    if isinstance(filters, (list, tuple)):
        if len(filters) != n:
            raise ValueError("one filter per file")
        return (C.c_int * n)(*(filter_code(f) for f in filters))
    return (C.c_int * n)(*([filter_code(filters)] * n))


def resize_center_crop(w, h, resize, crop, max_size=None):
    """torchvision's Resize(resize, max_size=max_size) followed by CenterCrop(crop) of a w x h PIL image, as the codec's
    resized size (W, H) and window (x, y, cw, ch).  resize: an int (the shorter side; the longer one is
    int(resize * long / short), capped by max_size) or torchvision's (h, w) sequence.  crop: an int or (h, w).  A crop larger
    than the resized image raises ValueError (torchvision pads it)."""
    if isinstance(resize, int) or len(resize) == 1:
        r = resize if isinstance(resize, int) else resize[0]
        short, long = (w, h) if w <= h else (h, w)
        new_short, new_long = r, int(r * long / short)
        if max_size is not None:
            if max_size <= r:
                raise ValueError(f"max_size = {max_size} must be strictly greater than the requested size {r}")
            if new_long > max_size:
                new_short, new_long = int(max_size * new_short / new_long), max_size
        W, H = (new_short, new_long) if w <= h else (new_long, new_short)
    else:
        if max_size is not None:
            raise ValueError("max_size applies only to an int resize")
        H, W = resize
    ch, cw = (crop, crop) if isinstance(crop, int) else (crop[0], crop[0]) if len(crop) == 1 else crop
    if cw > W or ch > H:
        raise ValueError(f"crop {cw}x{ch} is larger than the resized {W}x{H} image (torchvision would pad it)")
    return (W, H), (int(round((W - cw) / 2.0)), int(round((H - ch) / 2.0)), cw, ch)


DTYPES = {"uint8": 0, "float32": 1, "float16": 2, "bfloat16": 3}   # XPNGB_DT_*
DTYPE_BYTES = {"uint8": 1, "float32": 4, "float16": 2, "bfloat16": 2}
LAYOUTS = {"chw": 0, "hwc": 1}
SCALES = {"div": 0, "mul": 1}   # torchvision v1 to_tensor (x / 255), v2 ToDtype(scale=True) (x * (1 / 255))


def _dtype_name(dtype):
    """torch.float32 or "float32" -> "float32"."""
    name = dtype if isinstance(dtype, str) else str(dtype).removeprefix("torch.")
    if name not in DTYPES:
        raise ValueError(f"unsupported tensor dtype {dtype!r}: one of {sorted(DTYPES)}")
    return name


def tensor_format(dtype, layout="chw", scale="div", mean=(0, 0, 0, 0), std=(1, 1, 1, 1), drop_alpha=False):
    """The xpngb_tensor of a tensor decode.  dtype: torch.uint8 / float32 / float16 / bfloat16 (or its name); layout "chw" or
    "hwc"; scale "div" (torchvision's to_tensor) or "mul" (v2 ToDtype(scale=True)); mean and std per output channel (missing
    channels get mean 0, std 1); drop_alpha: 3 channels for RGBA files too, as PIL's convert("RGB")."""
    if layout not in LAYOUTS:
        raise ValueError(f"unknown layout {layout!r}")
    if scale not in SCALES:
        raise ValueError(f"unknown scale {scale!r}")
    mean, std = list(mean), list(std)
    if len(mean) > 4 or len(std) > 4:
        raise ValueError("at most 4 channels of mean and std")
    f = _Tensor()
    f.dtype, f.layout, f.scale, f.channels = DTYPES[_dtype_name(dtype)], LAYOUTS[layout], SCALES[scale], 3 if drop_alpha else 0
    f.mean[:] = [float(v) for v in mean + [0.0] * (4 - len(mean))]
    f.std[:] = [float(v) for v in std + [1.0] * (4 - len(std))]
    return f


def color_params(fn_idx, b, c, s, h, gray=False):
    """One entry's xpngb_color from T.ColorJitter.get_params(...)'s tuple as returned: fn_idx (a tensor or sequence of the
    step numbers 0 brightness, 1 contrast, 2 saturation, 3 hue, in the order applied) and the four factors, None for a
    step that is not applied.  gray: RandomGrayscale after the jitter."""
    col = _Color()
    col.order[:] = [int(k) for k in fn_idx]
    col.on = sum(1 << k for k, f in enumerate((b, c, s, h)) if f is not None)
    col.gray = int(bool(gray))
    col.factor[:] = [1.0 if b is None else float(b), 1.0 if c is None else float(c), 1.0 if s is None else float(s),
                     0.0 if h is None else float(h)]
    return col


def color_array(colors, n):
    """None, or one entry per file (color_params(...) or None for no colour) -> ctypes array of xpngb_color, or None."""
    if colors is None:
        return None
    if len(colors) != n:
        raise ValueError("one colour entry per file")
    arr = (_Color * n)()
    for i, c in enumerate(colors):
        if c is None:
            arr[i].order[:] = [0, 1, 2, 3]
        else:
            arr[i] = c
    return arr


def blur_params(radius=None, threshold=None):
    """One entry's xpngb_blur: radius, a number or (x, y), is ImageFilter.GaussianBlur's (None: no blur); threshold is
    ImageOps.solarize's after the blur (None: no solarize; 128 is ImageOps.solarize(img)'s default)."""
    b = _Blur()
    if radius is not None:
        b.radius[:] = [float(radius)] * 2 if isinstance(radius, (int, float)) else [float(r) for r in radius]
    if threshold is not None:
        b.solarize, b.threshold = 1, float(threshold)
    return b


def blur_array(blurs, n):
    """None, or one entry per file (blur_params(...) or None for neither step) -> ctypes array of xpngb_blur, or None."""
    if blurs is None:
        return None
    if len(blurs) != n:
        raise ValueError("one blur entry per file")
    arr = (_Blur * n)()
    for i, b in enumerate(blurs):
        if b is not None:
            arr[i] = b
    return arr


def blur_box(radius):
    """The library's (ri, ww, fw) of one axis of GaussianBlur(radius), as Pillow computes them; None for a refused radius."""
    ri, ww, fw = C.c_int32(), C.c_uint32(), C.c_uint32()
    if lib().xpngb_blur_box(float(radius), C.byref(ri), C.byref(ww), C.byref(fw)):
        return None
    return ri.value, ww.value, fw.value


AUG_KINDS = {"affine": 0, "transpose": 1, "brightness": 2, "color": 3, "contrast": 4, "sharpness": 5, "posterize": 6,
             "solarize": 7, "autocontrast": 8, "equalize": 9, "invert": 10}   # XPNGB_AUG_*
AUG_RESAMPLE = {"nearest": 0, "bilinear": 2, "bicubic": 3}                   # PIL.Image.Resampling numbers


def _inverse_affine(center, angle, translate, shear):
    """torchvision's _get_inverse_affine_matrix at scale 1, operation for operation."""
    rot, sx, sy = math.radians(angle), math.radians(shear[0]), math.radians(shear[1])
    cx, cy = center
    tx, ty = translate
    a = math.cos(rot - sy) / math.cos(sy)
    b = -math.cos(rot - sy) * math.tan(sx) / math.cos(sy) - math.sin(rot)
    c = math.sin(rot - sy) / math.cos(sy)
    d = -math.sin(rot - sy) * math.tan(sx) / math.cos(sy) + math.cos(rot)
    m = [x / 1.0 for x in (d, -b, 0.0, -c, a, 0.0)]
    m[2] += m[0] * (-cx - tx) + m[1] * (-cy - ty)
    m[5] += m[3] * (-cx - tx) + m[4] * (-cy - ty)
    m[2] += cx
    m[5] += cy
    return m


def _rotate_matrix(angle, w, h):
    """Image.rotate's matrix (no expand, centre (w / 2, h / 2)) for angle already reduced mod 360."""
    angle = -math.radians(angle)
    m = [round(math.cos(angle), 15), round(math.sin(angle), 15), 0.0, round(-math.sin(angle), 15), round(math.cos(angle), 15), 0.0]
    cx, cy = w / 2, h / 2
    m[2], m[5] = m[0] * (-cx - 0) + m[1] * (-cy - 0) + m[2], m[3] * (-cx - 0) + m[4] * (-cy - 0) + m[5]
    m[2] += cx
    m[5] += cy
    return m


def _resample_code(interpolation):
    if isinstance(interpolation, int):
        if interpolation not in AUG_RESAMPLE.values():
            raise ValueError(f"unknown augment resample {interpolation!r}: PIL NEAREST 0, BILINEAR 2 or BICUBIC 3")
        return int(interpolation)
    name = getattr(interpolation, "value", interpolation)
    if not isinstance(name, str) or name.lower() not in AUG_RESAMPLE:
        raise ValueError(f"unknown augment interpolation {interpolation!r}: one of {sorted(AUG_RESAMPLE)}")
    return AUG_RESAMPLE[name.lower()]


def augment_params(steps, size, interpolation="nearest", fill=None):
    """One entry's xpngb_augment: steps is a list of (op_name, magnitude) exactly as torchvision's
    transforms.autoaugment._apply_op receives them, size the entry's output (w, h) at that point of the pipeline.  The
    program is built as torchvision and Pillow build it in Python: _get_inverse_affine_matrix with torchvision's centres
    (0, 0 for the shears, the image centre otherwise), Image.rotate's angle % 360, its copy / 180 / square 90 and 270
    transposes and round(., 15), int(magnitude) for translate and posterize, 1 + magnitude factors and _parse_fill's int()."""
    w, h = int(size[0]), int(size[1])
    resample = _resample_code(interpolation)
    if fill is None:
        fill = 0
    if isinstance(fill, (int, float)):
        fill = (fill,) * 3
    fill = tuple(fill) * 3 if len(fill) == 1 else tuple(fill)
    if len(fill) != 3:
        raise ValueError("fill: one value or one per RGB channel")
    fill = tuple(int(v) for v in fill)
    if any(not 0 <= v <= 255 for v in fill):
        raise ValueError(f"fill {fill} is not a byte per channel")
    aug = _Augment()

    def add(kind, value=0.0, arg=0, data=None):
        if aug.nsteps == AUG_STEPS_MAX:
            raise ValueError(f"at most {AUG_STEPS_MAX} augment steps")
        s = aug.step[aug.nsteps]
        s.kind, s.value, s.arg = AUG_KINDS[kind], float(value), int(arg)
        if data is not None:
            s.data[:] = [float(v) for v in data]
            s.fill[:] = list(fill) + [0]
        aug.nsteps += 1

    for name, m in steps:
        if name == "ShearX":
            add("affine", arg=resample, data=_inverse_affine([0, 0], 0.0, [0, 0], [math.degrees(math.atan(m)), 0.0]))
        elif name == "ShearY":
            add("affine", arg=resample, data=_inverse_affine([0, 0], 0.0, [0, 0], [0.0, math.degrees(math.atan(m))]))
        elif name in ("TranslateX", "TranslateY"):
            t = [int(m), 0] if name == "TranslateX" else [0, int(m)]
            add("affine", arg=resample, data=_inverse_affine([w * 0.5, h * 0.5], 0.0, t, [0.0, 0.0]))
        elif name == "Rotate":
            a = m % 360.0
            if a == 0:
                continue
            if a == 180:
                add("transpose", arg=OPS["mvh"])
            elif a in (90, 270) and w == h:   # Transpose.ROTATE_90 turns counter-clockwise: r270
                add("transpose", arg=OPS["r270" if a == 90 else "r90"])
            else:
                add("affine", arg=resample, data=_rotate_matrix(a, w, h))
        elif name in ("Brightness", "Color", "Contrast", "Sharpness"):
            add(name.lower(), 1.0 + m)
        elif name == "Posterize":
            add("posterize", arg=int(m))
        elif name == "Solarize":
            add("solarize", m)
        elif name in ("AutoContrast", "Equalize", "Invert"):
            add(name.lower())
        elif name != "Identity":
            raise ValueError(f"unknown augment op {name!r}")
    return aug


def _replay_op(op_meta, name, magnitude_index, signed_draw):
    magnitudes, signed = op_meta[name]
    m = float(magnitudes[magnitude_index].item()) if magnitudes.ndim > 0 else 0.0
    return name, (-m if signed and signed_draw() else m)


def rand_augment_ops(ra, size):
    """The (op_name, magnitude) list one forward of torchvision's RandAugment module ra passes to _apply_op on a w x h = size
    image: its draws from torch's global RNG, in forward's order, with the module's own _augmentation_space."""
    import torch
    w, h = size
    op_meta = ra._augmentation_space(ra.num_magnitude_bins, (h, w))
    steps = []
    for _ in range(ra.num_ops):
        name = list(op_meta.keys())[int(torch.randint(len(op_meta), (1,)).item())]
        steps.append(_replay_op(op_meta, name, ra.magnitude, lambda: torch.randint(2, (1,))))
    return steps


def trivial_augment_wide_ops(ta, size):
    """The (op_name, magnitude) list of one forward of torchvision's TrivialAugmentWide module ta."""
    import torch
    op_meta = ta._augmentation_space(ta.num_magnitude_bins)
    name = list(op_meta.keys())[int(torch.randint(len(op_meta), (1,)).item())]
    magnitudes, _ = op_meta[name]
    idx = torch.randint(len(magnitudes), (1,), dtype=torch.long) if magnitudes.ndim > 0 else None
    return [_replay_op(op_meta, name, idx, lambda: torch.randint(2, (1,)))]


def auto_augment_ops(aa, size):
    """The (op_name, magnitude) list of one forward of torchvision's AutoAugment module aa (its own get_params and policies)."""
    w, h = size
    transform_id, probs, signs = aa.get_params(len(aa.policies))
    op_meta = aa._augmentation_space(10, (h, w))
    steps = []
    for i, (name, p, magnitude_id) in enumerate(aa.policies[transform_id]):
        if probs[i] <= p:
            magnitudes, signed = op_meta[name]
            m = float(magnitudes[magnitude_id].item()) if magnitude_id is not None else 0.0
            steps.append((name, -m if signed and signs[i] == 0 else m))
    return steps


def rand_augment_steps(ra, size):
    """The xpngb_augment of one forward of RandAugment module ra on a w x h = size image (rand_augment_ops' draws)."""
    return augment_params(rand_augment_ops(ra, size), size, ra.interpolation, ra.fill)


def trivial_augment_wide_steps(ta, size):
    """The xpngb_augment of one forward of TrivialAugmentWide module ta on a w x h = size image."""
    return augment_params(trivial_augment_wide_ops(ta, size), size, ta.interpolation, ta.fill)


def auto_augment_steps(aa, size):
    """The xpngb_augment of one forward of AutoAugment module aa on a w x h = size image."""
    return augment_params(auto_augment_ops(aa, size), size, aa.interpolation, aa.fill)


def augment_array(augs, n):
    """None, or one entry per file (augment_params(...) or None for no step) -> ctypes array of xpngb_augment, or None."""
    if augs is None:
        return None
    if len(augs) != n:
        raise ValueError("one augment entry per file")
    arr = (_Augment * n)()
    for i, a in enumerate(augs):
        if a is not None:
            arr[i] = a
    return arr


def region_tiles(w, h, rect):
    """Tiles a region decode of rect = (x, y, w, h) inside a w x h coded image decodes, and their union (x, y, w, h):
    (0, None) when rect is empty or not inside the image.  Host only."""
    r, cover = rects([rect])[0], _Rect()
    n = int(lib().xpngb_region_tiles(int(w), int(h), C.byref(r), C.byref(cover)))
    return n, ((cover.x, cover.y, cover.w, cover.h) if n else None)


class Codec:
    """One codec context on one CUDA device (one per process/rank)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        self.device = int(device)
        if lib().xpngb_create(C.byref(self._h), int(device)):
            raise RuntimeError("xpngb_create failed: no usable CUDA device (there is no CPU fallback)")
        # CUDA is initialised now: the queue count asked for in __init__.py has been read, children need not inherit it
        import xpng_b200 as _pkg
        if getattr(_pkg, "CONNECTIONS_SET_HERE", False):
            os.environ.pop("CUDA_DEVICE_MAX_CONNECTIONS", None)
            _pkg.CONNECTIONS_SET_HERE = False

    def close(self):
        if self._h:
            lib().xpngb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self):
        return lib().xpngb_last_error(self._h).decode()

    @property
    def last_kernel_ms(self):
        return float(lib().xpngb_last_kernel_ms(self._h))

    @property
    def last_launches(self):
        return int(lib().xpngb_last_launches(self._h))

    @property
    def last_tiles(self):
        """Tiles the last decode call decoded (stored files count 0; entries that share a file count its tiles once)."""
        return int(lib().xpngb_last_tiles(self._h))

    @property
    def stream(self):
        return lib().xpngb_stream(self._h)

    def profile(self, on):
        """Per-kernel CUDA-event timing (serialises launches); see profile_report()."""
        lib().xpngb_profile(self._h, 3 if on == 3 else int(bool(on)))   # 3: timeline to stderr, launches not serialised

    def profile_report(self):
        """{kernel name: (total ms, launches)} accumulated since profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        lib().xpngb_profile_report(self._h, buf, len(buf))
        out = {}
        for line in buf.value.decode().splitlines():
            name, ms, cnt = line.rsplit(" ", 2)
            out[name] = (float(ms), int(cnt))
        return out

    # ---------------------------------------------------------------- raw pointer API (bench / device-resident data)
    @staticmethod
    def layout(shapes):
        """[(h, w, c)] -> (descriptor array, total bytes): images packed at 16-byte aligned offsets."""
        arr = (_Image * len(shapes))()
        off = 0
        for i, (h, w, c) in enumerate(shapes):
            arr[i].w, arr[i].h, arr[i].offset, arr[i].A, arr[i].mode = w, h, off, int(c == 4), 0
            off = _align16(off + h * w * c)
        return arr, off

    def encode_raw(self, level, descs, n, pix_ptr, pix_size, pix_dev, out_ptr, out_cap, out_dev):
        offs, sizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
        if lib().xpngb_encode(self._h, int(level), descs, n, C.c_void_p(pix_ptr), pix_size, int(pix_dev),
                              C.c_void_p(out_ptr), out_cap, int(out_dev), offs, sizes):
            raise RuntimeError("xpngb_encode: " + self._err())
        return offs, sizes

    def decode_raw(self, descs, n, files_ptr, files_size, files_dev, offs, sizes, pix_ptr, pix_cap, pix_dev):
        if lib().xpngb_decode(self._h, descs, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs, sizes,
                              C.c_void_p(pix_ptr), pix_cap, int(pix_dev)):
            raise RuntimeError("xpngb_decode: " + self._err())

    def decode_region_raw(self, descs, rect_arr, n, files_ptr, files_size, files_dev, offs, sizes, pix_ptr, pix_cap, pix_dev):
        """decode_raw of rectangle rect_arr[i] (see rects()) of file i: crop i is written packed at pix_ptr + descs[i].offset."""
        if lib().xpngb_decode_region(self._h, descs, rect_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs, sizes,
                                     C.c_void_p(pix_ptr), pix_cap, int(pix_dev)):
            raise RuntimeError("xpngb_decode_region: " + self._err())

    def decode_oriented_raw(self, descs, ops_arr, rect_arr, n, files_ptr, files_size, files_dev, offs, sizes, pix_ptr, pix_cap, pix_dev):
        """decode_raw (rect_arr None) or decode_region_raw with entry i turned by ops_arr[i] (see op_codes()): written packed at
        pix_ptr + descs[i].offset, with width and height swapped for the quarter turns.  descs are not swapped."""
        if lib().xpngb_decode_oriented(self._h, ops_arr, descs, rect_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs,
                                       sizes, C.c_void_p(pix_ptr), pix_cap, int(pix_dev)):
            raise RuntimeError("xpngb_decode_oriented: " + self._err())

    def decode_resized_raw(self, descs, ops_arr, rect_arr, size_arr, n, files_ptr, files_size, files_dev, offs, sizes, pix_ptr, pix_cap,
                           pix_dev):
        """decode_oriented_raw with entry i resampled to size_arr[i] (see sizes()) before its op: Pillow's bilinear resize of the
        crop rect_arr[i] (None: whole images), ops_arr None for no op.  Written packed at pix_ptr + descs[i].offset as
        size_arr[i].h rows of size_arr[i].w pixels, swapped for the quarter turns."""
        if lib().xpngb_decode_resized(self._h, ops_arr, descs, rect_arr, size_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev),
                                      offs, sizes, C.c_void_p(pix_ptr), pix_cap, int(pix_dev)):
            raise RuntimeError("xpngb_decode_resized: " + self._err())

    def decode_tensor_raw(self, fmt, descs, ops_arr, rect_arr, size_arr, n, files_ptr, files_size, files_dev, offs, sizes, out_ptr,
                          out_cap, out_dev):
        """decode_resized_raw (size_arr None: no resize, as decode_oriented_raw) with entry i written as a tensor of format fmt
        (see tensor_format()) at out_ptr + descs[i].offset: C * H * W elements, H and W after the op."""
        if lib().xpngb_decode_tensor(self._h, C.byref(fmt), ops_arr, descs, rect_arr, size_arr, n, C.c_void_p(files_ptr), files_size,
                                     int(files_dev), offs, sizes, C.c_void_p(out_ptr), out_cap, int(out_dev)):
            raise RuntimeError("xpngb_decode_tensor: " + self._err())

    def decode_resampled_raw(self, fmt, descs, filt_arr, ops_arr, rect_arr, size_arr, win_arr, n, files_ptr, files_size, files_dev,
                             offs, sizes, out_ptr, out_cap, out_dev):
        """decode_resized_raw (fmt None) or decode_tensor_raw with entry i resampled by filt_arr[i] (see filter_codes(); None:
        bilinear) and only window win_arr[i] (see rects(), in size_arr[i]'s coordinates; None: all of it) written, as
        win_arr[i].h rows of win_arr[i].w pixels (or tensor elements), swapped for the quarter turns."""
        if lib().xpngb_decode_resampled(self._h, None if fmt is None else C.byref(fmt), filt_arr, ops_arr, descs, rect_arr, size_arr,
                                        win_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs, sizes, C.c_void_p(out_ptr),
                                        out_cap, int(out_dev)):
            raise RuntimeError("xpngb_decode_resampled: " + self._err())

    def decode_color_raw(self, fmt, descs, filt_arr, ops_arr, rect_arr, size_arr, win_arr, color_arr, n, files_ptr, files_size, files_dev,
                         offs, sizes, out_ptr, out_cap, out_dev):
        """decode_resampled_raw (size_arr None: no resize, filt_arr and win_arr then None, as decode_tensor_raw /
        decode_oriented_raw) with ColorJitter and RandomGrayscale color_arr[i] (see color_array(); None: none) applied to
        entry i's pixels before they are written."""
        if lib().xpngb_decode_color(self._h, None if fmt is None else C.byref(fmt), filt_arr, ops_arr, descs, rect_arr, size_arr, win_arr,
                                    color_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs, sizes, C.c_void_p(out_ptr),
                                    out_cap, int(out_dev)):
            raise RuntimeError("xpngb_decode_color: " + self._err())

    def decode_blur_raw(self, fmt, descs, filt_arr, ops_arr, rect_arr, size_arr, win_arr, color_arr, blur_arr, n, files_ptr, files_size,
                        files_dev, offs, sizes, out_ptr, out_cap, out_dev):
        """decode_color_raw (color_arr None: no colour) with GaussianBlur and solarize blur_arr[i] (see blur_array(); None:
        none) applied to entry i's pixels after its colour step."""
        if lib().xpngb_decode_blur(self._h, None if fmt is None else C.byref(fmt), filt_arr, ops_arr, descs, rect_arr, size_arr, win_arr,
                                   color_arr, blur_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs, sizes,
                                   C.c_void_p(out_ptr), out_cap, int(out_dev)):
            raise RuntimeError("xpngb_decode_blur: " + self._err())

    def decode_augment_raw(self, fmt, descs, filt_arr, ops_arr, rect_arr, size_arr, win_arr, color_arr, blur_arr, aug_arr, n, files_ptr,
                           files_size, files_dev, offs, sizes, out_ptr, out_cap, out_dev):
        """decode_blur_raw (blur_arr None: no blur) with the augment program aug_arr[i] (see augment_array(); None: none) run
        on entry i's pixels right after its op, before its colour step."""
        if lib().xpngb_decode_augment(self._h, None if fmt is None else C.byref(fmt), filt_arr, ops_arr, descs, rect_arr, size_arr,
                                      win_arr, color_arr, blur_arr, aug_arr, n, C.c_void_p(files_ptr), files_size, int(files_dev), offs,
                                      sizes, C.c_void_p(out_ptr), out_cap, int(out_dev)):
            raise RuntimeError("xpngb_decode_augment: " + self._err())

    def resize_coeffs(self, filt, inn, out, first=0, count=None):
        """The device's weight tables of an inn -> out axis for output coordinates first .. first + count - 1: (xmin, n) as
        an (count, 2) int32 array and the (count, ksize) int32 weights, zero past each window."""
        f = filter_code(filt)
        count = out - first if count is None else count
        ksize = int(lib().xpngb_resize_ksize(f, inn, out))
        xn = np.zeros((max(count, 1), 2), np.int32)
        k = np.zeros((max(count, 1), max(ksize, 1)), np.int32)
        if lib().xpngb_resize_coeffs(self._h, f, inn, out, first, count, xn.ctypes.data_as(C.POINTER(C.c_int32)),
                                     k.ctypes.data_as(C.POINTER(C.c_int32))):
            raise RuntimeError("xpngb_resize_coeffs: " + self._err())
        return xn[:count], k[:count, :ksize]

    def decode_tensor(self, files, sizes=None, boxes=None, ops=None, dtype=None, layout="chw", scale="div", mean=None, std=None,
                      drop_alpha=False, filters=None, windows=None, colors=None, blurs=None, augments=None):
        """list of .xpng byte strings -> one torch tensor on this codec's device, (N, C, H, W) for layout "chw" or (N, H, W, C)
        for "hwc": each whole image, or rectangle boxes[i] = (x, y, w, h) of it, resized to sizes[i] = (w, h) as decode_resized
        does (None: not resized), turned by ops[i] (None: no op), then scaled and normalised as torchvision does, bit for bit:
        scale "div" is F.normalize(F.to_tensor(pil), mean, std), "mul" is v2.Normalize after v2.ToDtype(float32, scale=True);
        float16 / bfloat16 are those results rounded by .to(dtype).  dtype: torch.float32 (default), float16, bfloat16 or
        uint8 (the bytes themselves, as F.pil_to_tensor).  mean / std None: 0 and 1 (no Normalize).  C is 3 + A, or 3 with
        drop_alpha.  filters and windows (only with sizes) as decode_resized: torchvision's Resize(256) + CenterCrop(224) of
        each image is sizes[i], windows[i] = resize_center_crop(w, h, 256, 224).  colors: one color_params(...) or None per
        entry, ColorJitter and RandomGrayscale applied before the conversion (sizes not needed).  blurs: one blur_params(...) or
        None per entry, GaussianBlur and solarize applied after the colour step (sizes not needed).  augments: one
        augment_params(...) (or rand_augment_steps / trivial_augment_wide_steps / auto_augment_steps) or None per entry, run
        right after the op, before the colour step (sizes not needed).  Every entry must have the same output shape (ValueError
        otherwise); ragged batches use decode_tensor_raw, decode_resampled_raw, decode_color_raw, decode_blur_raw or
        decode_augment_raw."""
        import torch
        n = len(files)
        if n == 0:
            raise ValueError("decode_tensor needs at least one file")
        for name, arg in (("size", sizes), ("rectangle", boxes), ("op", ops), ("window", windows), ("colour entry", colors),
                          ("blur entry", blurs), ("augment entry", augments)):
            if arg is not None and len(arg) != n:
                raise ValueError(f"one {name} per file")
        if sizes is None and (filters is not None or windows is not None):
            raise ValueError("filters and windows need sizes")
        dname = _dtype_name(torch.float32 if dtype is None else dtype)
        fmt = tensor_format(dname, layout, scale, (0, 0, 0, 0) if mean is None else mean, (1, 1, 1, 1) if std is None else std, drop_alpha)
        ra = None if boxes is None else rects(boxes)
        sa = None if sizes is None else _sizes(sizes)
        wa = None if windows is None else rects(windows)
        fa = filter_codes(filters, n)
        descs, foffs, fsizes, fb, off, _, _ = self._pack_files(files, ra, sa)
        shapes = set()
        for i, d in enumerate(descs):
            w, h = (wa[i].w, wa[i].h) if wa is not None else (sa[i].w, sa[i].h) if sa is not None else (ra[i].w, ra[i].h) if ra is not None else (d.w, d.h)
            if ops is not None and ops[i] in QUARTER_TURNS:
                w, h = h, w
            shapes.add((3 if drop_alpha else 3 + d.A, h, w))
        if len(shapes) != 1:
            raise ValueError(f"entries have different output shapes {sorted(shapes)}: use decode_tensor_raw for ragged batches")
        c, h, w = shapes.pop()
        per = c * h * w
        stride = _align16(per * DTYPE_BYTES[dname]) // DTYPE_BYTES[dname]   # entry offsets are multiples of 16 bytes
        for i in range(n):
            descs[i].offset = i * stride * DTYPE_BYTES[dname]
        dev = torch.device("cuda", self.device)
        flat = torch.empty(n * stride, dtype=getattr(torch, dname), device=dev)
        # the library writes on its own stream: memory fresh from the caching allocator may still be in use by queued work
        torch.cuda.current_stream(dev).synchronize()
        oa = None if ops is None else op_codes(ops)
        if augments is not None:
            self.decode_augment_raw(fmt, descs, fa, oa, ra, sa, wa, color_array(colors, n), blur_array(blurs, n), augment_array(augments, n),
                                    n, fb.ctypes.data, off, 0, foffs, fsizes, flat.data_ptr(), n * stride * DTYPE_BYTES[dname], 1)
        elif blurs is not None:
            self.decode_blur_raw(fmt, descs, fa, oa, ra, sa, wa, color_array(colors, n), blur_array(blurs, n), n, fb.ctypes.data, off, 0,
                                 foffs, fsizes, flat.data_ptr(), n * stride * DTYPE_BYTES[dname], 1)
        elif colors is not None:
            self.decode_color_raw(fmt, descs, fa, oa, ra, sa, wa, color_array(colors, n), n, fb.ctypes.data, off, 0, foffs, fsizes,
                                  flat.data_ptr(), n * stride * DTYPE_BYTES[dname], 1)
        elif fa is None and wa is None:
            self.decode_tensor_raw(fmt, descs, oa, ra, sa, n, fb.ctypes.data, off, 0, foffs, fsizes, flat.data_ptr(),
                                   n * stride * DTYPE_BYTES[dname], 1)
        else:
            self.decode_resampled_raw(fmt, descs, fa, oa, ra, sa, wa, n, fb.ctypes.data, off, 0, foffs, fsizes, flat.data_ptr(),
                                      n * stride * DTYPE_BYTES[dname], 1)
        out = flat.view(n, stride)[:, :per]
        out = out.reshape(n, c, h, w) if layout == "chw" else out.reshape(n, h, w, c)
        return out.contiguous()

    VIEW_KEYS = ("sizes", "boxes", "ops", "filters", "windows", "colors", "blurs", "augments")

    def decode_views(self, files, views, dtype=None, layout="chw", scale="div", mean=None, std=None, drop_alpha=False):
        """Every view of a multi-crop batch from one library call: a list of V tensors on this codec's device, view v of
        shape (N, C, h_v, w_v) (or (N, h_v, w_v, C) for layout "hwc"), as decode_tensor(files, **views[v], dtype=dtype, ...)
        returns it, bit for bit.  views: V dicts, each holding decode_tensor's per-entry arguments for one view of every
        file (keys VIEW_KEYS: sizes, boxes, ops, filters, windows, colors, blurs, augments; a missing key is decode_tensor's
        None).  Different views may have different shapes (DINO's 224 and 96); the entries of one view must share one
        (ValueError naming the view otherwise).  Each file is packed and uploaded once, and the library decodes the tiles of
        each file once for all its views: the bounding box of the tiles its views' rectangles touch."""
        import torch
        n, nv = len(files), len(views)
        if n == 0 or nv == 0:
            raise ValueError("decode_views needs at least one file and one view")
        for v, d in enumerate(views):
            bad = sorted(set(d) - set(self.VIEW_KEYS))
            if bad:
                raise ValueError(f"view {v}: unknown key {bad[0]!r} (one of {', '.join(self.VIEW_KEYS)})")
            for k in ("sizes", "boxes", "ops", "windows", "colors", "blurs", "augments"):
                if d.get(k) is not None and len(d[k]) != n:
                    raise ValueError(f"view {v}: one {k[:-1] if k != 'boxes' else 'box'} per file")
            if d.get("sizes") is None and (d.get("filters") is not None or d.get("windows") is not None):
                raise ValueError(f"view {v}: filters and windows need sizes")
        heads = []
        for i, f in enumerate(files):
            d = _Image()
            if lib().xpngb_peek(np.frombuffer(f, dtype=np.uint8).ctypes.data, len(f), C.byref(d)):
                raise ValueError(f"file {i}: not an .xpng header")
            heads.append(d)
        # entry v * n + i is view v of file i; a view without some argument gets the value that leaves its entries as
        # decode_tensor leaves them without it (an output size equal to the crop is no resize)
        any_of = {k: any(d.get(k) is not None for d in views) for k in self.VIEW_KEYS}
        boxes, szs, wins, ops, filt, cols, bls, augs, shapes = [], [], [], [], [], [], [], [], []
        for v, d in enumerate(views):
            try:
                fc = filter_codes(d.get("filters"), n)
            except ValueError as e:
                raise ValueError(f"view {v}: {e}") from None
            shape = set()
            for i in range(n):
                b = d["boxes"][i] if d.get("boxes") is not None else (0, 0, heads[i].w, heads[i].h)
                z = d["sizes"][i] if d.get("sizes") is not None else (b[2], b[3])
                wn = d["windows"][i] if d.get("windows") is not None else (0, 0, z[0], z[1])
                op = d["ops"][i] if d.get("ops") is not None else "tl"
                boxes.append(b); szs.append(z); wins.append(wn); ops.append(op)
                filt.append(FILTERS["bilinear"] if fc is None else fc[i])
                cols.append(d["colors"][i] if d.get("colors") is not None else None)
                bls.append(d["blurs"][i] if d.get("blurs") is not None else None)
                augs.append(d["augments"][i] if d.get("augments") is not None else None)
                w, h = int(wn[2]), int(wn[3])
                shape.add((3 if drop_alpha else 3 + heads[i].A,) + ((w, h) if op in QUARTER_TURNS else (h, w)))
            if len(shape) != 1:
                raise ValueError(f"view {v}: entries have different output shapes {sorted(shape)}")
            shapes.append(shape.pop())
        m = n * nv
        dname = _dtype_name(torch.float32 if dtype is None else dtype)
        fmt = tensor_format(dname, layout, scale, (0, 0, 0, 0) if mean is None else mean, (1, 1, 1, 1) if std is None else std, drop_alpha)
        ra = rects(boxes) if any_of["boxes"] else None
        sa = _sizes(szs) if any_of["sizes"] else None
        wa = rects(wins) if any_of["windows"] else None
        descs, foffs, fsizes, fb, off, _, _ = self._pack_files(list(files) * nv, ra, sa)
        eb = DTYPE_BYTES[dname]
        bases, strides, at = [], [], 0
        for c, h, w in shapes:
            stride = _align16(c * h * w * eb) // eb   # entry offsets are multiples of 16 bytes
            bases.append(at)
            strides.append(stride)
            at += n * stride
        for v in range(nv):
            for i in range(n):
                descs[v * n + i].offset = (bases[v] + i * strides[v]) * eb
        dev = torch.device("cuda", self.device)
        flat = torch.empty(at, dtype=getattr(torch, dname), device=dev)
        # the library writes on its own stream: memory fresh from the caching allocator may still be in use by queued work
        torch.cuda.current_stream(dev).synchronize()
        self.decode_augment_raw(fmt, descs, (C.c_int * m)(*filt) if any_of["filters"] else None, op_codes(ops) if any_of["ops"] else None,
                                ra, sa, wa, color_array(cols, m) if any_of["colors"] else None,
                                blur_array(bls, m) if any_of["blurs"] else None, augment_array(augs, m) if any_of["augments"] else None,
                                m, fb.ctypes.data, off, 0, foffs, fsizes, flat.data_ptr(), at * eb, 1)
        out = []
        for v, (c, h, w) in enumerate(shapes):
            t = flat[bases[v]: bases[v] + n * strides[v]].view(n, strides[v])[:, :c * h * w]
            out.append((t.reshape(n, c, h, w) if layout == "chw" else t.reshape(n, h, w, c)).contiguous())
        return out

    # ---------------------------------------------------------------- numpy convenience (host buffers)
    def encode(self, level, images):
        """list of (h,w,3|4) uint8 arrays -> list of .xpng byte strings."""
        images = [np.ascontiguousarray(a, dtype=np.uint8) for a in images]
        descs, total = self.layout([a.shape for a in images])
        buf = np.zeros(total + 16, dtype=np.uint8)
        for d, a in zip(descs, images):
            buf[d.offset: d.offset + a.size] = a.reshape(-1)
        cap = int(lib().xpngb_encode_bound(descs, len(images)))
        out = np.empty(cap + 16, dtype=np.uint8)
        offs, sizes = self.encode_raw(level, descs, len(images), buf.ctypes.data, total, 0, out.ctypes.data, cap, 0)
        return [out[offs[i]: offs[i] + sizes[i]].tobytes() for i in range(len(images))]

    def _pack_files(self, files, ra=None, sa=None, wa=None):
        """Files packed at 16-byte offsets and a host output buffer: one whole image, crop ra[i], size sa[i] or window wa[i]
        per entry.  An object that appears in several entries is packed once: those entries share its offset, so the
        library decodes it once for all of them."""
        n = len(files)
        descs = (_Image * n)()
        foffs, fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
        off = poff = 0
        packed = {}   # id(file) -> offset
        for i, f in enumerate(files):
            b = np.frombuffer(f, dtype=np.uint8)
            if lib().xpngb_peek(b.ctypes.data, len(f), C.byref(descs[i])):
                raise ValueError(f"file {i}: not an .xpng header")
            if id(f) in packed:
                foffs[i], fsizes[i] = packed[id(f)], len(f)
            else:
                packed[id(f)] = foffs[i] = off
                fsizes[i] = len(f)
                off = _align16(off + len(f))
            descs[i].offset = poff
            if wa is not None:
                if 0 < wa[i].w <= 1 << 24 and 0 < wa[i].h <= 1 << 24:   # other windows are refused by the library, naming the entry
                    poff = _align16(poff + wa[i].w * wa[i].h * (3 + descs[i].A))
            elif sa is not None:
                if 0 < sa[i].w <= 1 << 24 and 0 < sa[i].h <= 1 << 24:   # other sizes are refused by the library, naming the entry
                    poff = _align16(poff + sa[i].w * sa[i].h * (3 + descs[i].A))
            elif ra is None:
                poff = _align16(poff + descs[i].w * descs[i].h * (3 + descs[i].A))
            elif ra[i].w <= descs[i].w and ra[i].h <= descs[i].h:     # other rectangles are refused by the library, naming the entry
                poff = _align16(poff + ra[i].w * ra[i].h * (3 + descs[i].A))
        fb = np.zeros(off + 16, dtype=np.uint8)
        for f in {id(f): f for f in files}.values():
            fb[packed[id(f)]: packed[id(f)] + len(f)] = np.frombuffer(f, dtype=np.uint8)
        px = np.empty(poff + 16, dtype=np.uint8)
        return descs, foffs, fsizes, fb, off, px, poff

    @staticmethod
    def _unpack(px, descs, sizes, ops):
        """Entry i of px as an (h, w, c) array, w x h = sizes[i]; (w, h, c) for the quarter turns of ops."""
        out = []
        for i, (d, (w, h)) in enumerate(zip(descs, sizes)):
            c = 3 + d.A
            if ops is not None and ops[i] in QUARTER_TURNS:
                w, h = h, w
            out.append(px[d.offset: d.offset + w * h * c].reshape(h, w, c).copy())
        return out

    def decode(self, files, ops=None):
        """list of .xpng byte strings -> list of (h,w,3|4) uint8 arrays.  ops: one OPS name per file, each image written as
        that op leaves it ((w,h,3|4) for 'r90' and 'r270'); inverse_op(op) restores files written by encode_oriented(op)."""
        n = len(files)
        if ops is not None and len(ops) != n:
            raise ValueError("one op per file")
        descs, foffs, fsizes, fb, off, px, poff = self._pack_files(files)
        if ops is None:
            self.decode_raw(descs, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        else:
            self.decode_oriented_raw(descs, op_codes(ops), None, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        return self._unpack(px, descs, [(d.w, d.h) for d in descs], ops)

    def decode_region(self, files, boxes, ops=None):
        """list of .xpng byte strings and one (x, y, w, h) rectangle per file -> list of (h, w, 3|4) uint8 crops.  Only the
        tiles a rectangle touches are decoded; the same file may appear several times.  ops: one OPS name per entry, applied
        to the crop (rectangles are in the file's coordinates); 'r90' and 'r270' crops come back as (w, h, 3|4)."""
        n = len(files)
        if len(boxes) != n:
            raise ValueError("one rectangle per file")
        if ops is not None and len(ops) != n:
            raise ValueError("one op per file")
        ra = rects(boxes)
        descs, foffs, fsizes, fb, off, px, poff = self._pack_files(files, ra)
        if ops is None:
            self.decode_region_raw(descs, ra, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        else:
            self.decode_oriented_raw(descs, op_codes(ops), ra, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        return self._unpack(px, descs, [(r.w, r.h) for r in ra], ops)

    def decode_resized(self, files, sizes, boxes=None, ops=None, filters=None, windows=None, colors=None, blurs=None, augments=None):
        """list of .xpng byte strings and one (w, h) output size per file -> list of (h, w, 3|4) uint8 arrays: each whole image,
        or rectangle boxes[i] = (x, y, w, h) of it, resampled as Pillow's Image.resize((w, h), filter) does, every channel on
        its own (alpha is not premultiplied).  filters: None (bilinear), one filter for all entries or one per entry, each a
        name ("bicubic", ...), a PIL.Image.Resampling value or a torchvision InterpolationMode.  windows: one (x, y, w, h) per
        entry in the resized image's coordinates, the part of it that is returned (None: all of it).  ops: one OPS name per
        entry, applied last; 'r90' and 'r270' entries come back as (w, h, 3|4).  An entry whose size equals its crop is the
        crop itself.  colors: one color_params(...) or None per entry, ColorJitter and RandomGrayscale applied to its pixels.
        blurs: one blur_params(...) or None per entry, GaussianBlur and solarize applied to its pixels after the colour step.
        augments: one augment_params(...) or None per entry, run on its pixels right after the op, before the colour step."""
        n = len(files)
        if len(sizes) != n:
            raise ValueError("one size per file")
        if boxes is not None and len(boxes) != n:
            raise ValueError("one rectangle per file")
        if ops is not None and len(ops) != n:
            raise ValueError("one op per file")
        if windows is not None and len(windows) != n:
            raise ValueError("one window per file")
        ca = color_array(colors, n)
        ba = blur_array(blurs, n)
        aa = augment_array(augments, n)
        ra = None if boxes is None else rects(boxes)
        sa = _sizes(sizes)
        wa = None if windows is None else rects(windows)
        fa = filter_codes(filters, n)
        oa = None if ops is None else op_codes(ops)
        descs, foffs, fsizes, fb, off, px, poff = self._pack_files(files, ra, sa, wa)
        if aa is not None:
            self.decode_augment_raw(None, descs, fa, oa, ra, sa, wa, ca, ba, aa, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data,
                                    poff, 0)
        elif ba is not None:
            self.decode_blur_raw(None, descs, fa, oa, ra, sa, wa, ca, ba, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        elif ca is not None:
            self.decode_color_raw(None, descs, fa, oa, ra, sa, wa, ca, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        elif fa is None and wa is None:
            self.decode_resized_raw(descs, oa, ra, sa, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        else:
            self.decode_resampled_raw(None, descs, fa, oa, ra, sa, wa, n, fb.ctypes.data, off, 0, foffs, fsizes, px.ctypes.data, poff, 0)
        return self._unpack(px, descs, [(z.w, z.h) for z in (sa if wa is None else wa)], ops)

    # ---------------------------------------------------------------- traversal-order operations (Mirroring_and_Rotating/tool.c)
    def _pack(self, images):
        images = [np.ascontiguousarray(a, dtype=np.uint8) for a in images]
        descs, total = self.layout([a.shape for a in images])
        buf = np.zeros(total + 16, dtype=np.uint8)
        for d, a in zip(descs, images):
            buf[d.offset: d.offset + a.size] = a.reshape(-1)
        return images, descs, total, buf

    def transform(self, op, images):
        """Apply op ('r90', 'r270', 'mv', 'mh', 'mvh', 'tl', 'tr' — tool.c:133) to a list of (h,w,3|4) arrays."""
        images, descs, total, buf = self._pack(images)
        out = np.empty(total + 16, dtype=np.uint8)
        if lib().xpngb_transform(self._h, OPS[op], descs, len(images), buf.ctypes.data, total, 0, out.ctypes.data, 0):
            raise RuntimeError("xpngb_transform: " + self._err())
        return [out[d.offset: d.offset + d.w * d.h * (3 + d.A)].reshape(d.h, d.w, 3 + d.A).copy() for d in descs]

    def encode_oriented(self, level, op, images):
        """.xpng files of the images as `op` would leave them (tool --op followed by xpng -level), pixels untouched."""
        images, descs, total, buf = self._pack(images)
        n = len(images)
        cap = int(lib().xpngb_encode_bound(descs, n))
        out = np.empty(cap + 16, dtype=np.uint8)
        offs, sizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
        if lib().xpngb_encode_oriented(self._h, int(level), OPS[op], descs, n, buf.ctypes.data, total, 0, out.ctypes.data, cap, 0,
                                       offs, sizes):
            raise RuntimeError("xpngb_encode_oriented: " + self._err())
        return [out[offs[i]: offs[i] + sizes[i]].tobytes() for i in range(n)]

    def ycocg_forward(self, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(-1, 3)
        out = np.empty((len(rgb), 3), dtype=np.int16)
        if lib().xpngb_ycocg_forward(self._h, rgb.ctypes.data, out.ctypes.data, len(rgb)):
            raise RuntimeError(self._err())
        return out

    def ycocg_inverse(self, ycc):
        ycc = np.ascontiguousarray(ycc, dtype=np.int16).reshape(-1, 3)
        out = np.empty((len(ycc), 3), dtype=np.uint8)
        if lib().xpngb_ycocg_inverse(self._h, ycc.ctypes.data, out.ctypes.data, len(ycc)):
            raise RuntimeError(self._err())
        return out


# ---------------------------------------------------------------- reference-shaped file API (xpng.h / seven.h)

def _as_xpng(px):
    px = np.ascontiguousarray(px, dtype=np.uint8)
    h, w, c = px.shape
    return _Xpng(px.ctypes.data, w, h, px.size, c == 4), px


def xpng_store(mode, px, path):
    """xpng_store(mode, pm, path) of xpng.h:12 — returns False on success (the reference's 0)."""
    pm, keep = _as_xpng(px)
    return bool(lib().xpng_store(int(mode), C.byref(pm), os.fsencode(path)))


def _take(pm):
    c = 3 + int(pm.A)
    arr = np.ctypeslib.as_array(C.cast(pm.p, C.POINTER(C.c_uint8)), shape=(pm.s,)).reshape(pm.h, pm.w, c).copy()
    C.CDLL(None).free(C.c_void_p(pm.p))
    return arr


def xpng_load(path):
    """xpng_load(path, &pm) of xpng.h:13 — returns the pixels or raises."""
    pm = _Xpng()
    if lib().xpng_load(os.fsencode(path), C.byref(pm)):
        raise RuntimeError("xpng_load failed")
    return _take(pm)


def store_7(px, path):
    pm, keep = _as_xpng(px)
    return bool(lib().store_7(C.byref(pm), os.fsencode(path)))


def load_7(path):
    pm = _Xpng()
    if lib().load_7(os.fsencode(path), C.byref(pm)):
        raise RuntimeError("load_7 failed")
    return _take(pm)
