#!/usr/bin/env python
"""Colour decode on the GPU; one JSON line to profiles/color_decode_<tag>.json.  Files and outputs in device memory.

The workload is a BYOL-style training batch: sintel-like 1080p frames at levels 1 and 2, each with a seeded
RandomResizedCrop box resized (bilinear) to 224 x 224, a horizontal flip with p 0.5, ColorJitter(0.4, 0.4, 0.2, 0.1) with p 0.8
and RandomGrayscale with p 0.2, written as an ImageNet-normalised float32 (N, 3, 224, 224) tensor.  The arms, called in turn:
  floor   tensor decode of the same boxes and flips without colour (xpngb_decode_resampled)
  color   the whole transform in one xpngb_decode_color call
  tv_gpu  uint8 decode (xpngb_decode_resized), then torchvision's tensor ops on the GPU per entry, then ToDtype + Normalize;
          its byte mismatch rate against tests/test_color_decode.py's color_ref is reported
A sample of the colour arm is compared with color_ref first.  Each timing is 3 warm-up calls, then --reps calls per arm, each
ending in a device synchronise; the median is reported.  Per-kernel times of one colour call come from xpngb_profile.
Usage: python tools/color_decode_bench.py [--frames 1000] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, color_array, color_params, op_codes, rects, sizes, tensor_format  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import rrc_boxes  # noqa: E402
from test_resampled_decode import resize_pil  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from test_color_decode import color_ref  # noqa: E402
from resampled_decode_bench import alternate  # noqa: E402

OUT = (224, 224)
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def programs(n, seed):
    """Flip and colour entry per frame, drawn as RandomHorizontalFlip, RandomApply([ColorJitter], 0.8) and RandomGrayscale do."""
    import torchvision.transforms as T
    cj = T.ColorJitter(0.4, 0.4, 0.2, 0.1)
    torch.manual_seed(seed)
    ops, cols = [], []
    for _ in range(n):
        ops.append("mh" if torch.rand(1) < 0.5 else "tl")
        p = cj.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue) if not (0.8 < torch.rand(1)) else None
        gray = bool(torch.rand(1) < 0.2)
        cols.append(None if p is None and not gray else color_params(*(p or ([0, 1, 2, 3], None, None, None, None)), gray=gray))
    return ops, cols


def tv_apply(t, c):
    """torchvision's tensor-path ColorJitter + RandomGrayscale of one uint8 (3, H, W) GPU tensor for colour entry c."""
    import torchvision.transforms.functional as F
    if c is None:
        return t
    fns = (F.adjust_brightness, F.adjust_contrast, F.adjust_saturation, F.adjust_hue)
    for k in c.order:
        if (c.on >> k) & 1:
            t = fns[k](t, c.factor[k])
    return F.rgb_to_grayscale(t, 3) if c.gray else t


def run_level(cd, files, boxes, ops, cols, reps):
    n = len(files)
    B = Batch(files)
    fptr = B.dev.data_ptr()
    ra, sa, oa, ca = rects(boxes), sizes([OUT] * n), op_codes(ops), color_array(cols, n)
    fmt = tensor_format("float32", "chw", "div", MEAN, STD, drop_alpha=True)
    per = 3 * OUT[0] * OUT[1]
    td = (_Image * n)()
    for i in range(n):
        td[i].offset = i * per * 4
    t_floor = torch.empty((n, 3, *OUT[::-1]), dtype=torch.float32, device="cuda")
    t_col = torch.empty_like(t_floor)
    u8 = torch.empty((n, OUT[1], OUT[0], 3), dtype=torch.uint8, device="cuda")
    ud = (_Image * n)()
    for i in range(n):
        ud[i].offset = i * per
    mean = torch.tensor(MEAN, device="cuda").view(3, 1, 1)
    std = torch.tensor(STD, device="cuda").view(3, 1, 1)

    floor = lambda: cd.decode_resampled_raw(fmt, td, None, oa, ra, sa, None, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t_floor.data_ptr(), n * per * 4, 1)
    color = lambda: cd.decode_color_raw(fmt, td, None, oa, ra, sa, None, ca, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t_col.data_ptr(), n * per * 4, 1)

    def tv_u8():
        cd.decode_resized_raw(ud, oa, ra, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u8.data_ptr(), n * per, 1)
        return [tv_apply(u8[i].permute(2, 0, 1), cols[i]) for i in range(n)]

    def tv_gpu():
        out = torch.stack(tv_u8()).float().div_(255).sub_(mean).div_(std)
        return out

    # correctness of the colour arm on a sample, and the tensor path's mismatch rate
    color(); torch.cuda.synchronize()
    u = tv_u8(); torch.cuda.synchronize()
    base = u8.cpu().numpy()                     # uint8 decode without colour (resized, flipped)
    diff = total = 0
    for i in range(0, n, max(1, n // 40)):
        x, y, w, h = boxes[i]
        full = po.decode(files[i])
        px = po.orient(ops[i], resize_pil(full[y: y + h, x: x + w], *OUT, 2))
        if not np.array_equal(px, base[i]):
            raise SystemExit(f"entry {i}: the uint8 decode differs from the reference")
        want = px if cols[i] is None else color_ref(px, cols[i])
        if not np.array_equal(bits(t_col[i]), to_tensor_ref(want, "float32", "chw", "div", MEAN, STD)):
            raise SystemExit(f"entry {i}: colour decode differs from color_ref")
        tv = u[i].permute(1, 2, 0).cpu().numpy()
        diff += int((tv != want).sum()); total += want.size
    cd.profile(True)
    color()
    prof = {k: v for k, v in cd.profile_report().items() if k.startswith("k_color") or k == "k_to_tensor"}
    cd.profile(False)
    r = alternate({"floor_tensor_no_colour": floor, "color_decode": color, "tv_gpu_tensor_ops": tv_gpu}, reps)
    r["tv_gpu_mismatch_bytes_vs_color_ref"] = round(diff / total, 4)
    r["profiled_one_call_ms"] = {k: round(v[0], 3) for k, v in prof.items()}
    r["coloured_entries"] = sum(c is not None for c in cols)
    del B
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/color_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("color_decode_bench needs a CUDA device")
    res = {"tool": "tools/color_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "frames": a.frames, "size": list(OUT)}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    boxes = rrc_boxes(np.random.default_rng(2029), len(frames))
    ops, cols = programs(len(frames), 2030)
    for lv in (1, 2):
        files = []
        for k in range(0, len(frames), 250):
            files += cd.encode(lv, frames[k: k + 250])
        res[f"byol_224_f32_L{lv}"] = run_level(cd, files, boxes, ops, cols, a.reps)
        print(json.dumps(res[f"byol_224_f32_L{lv}"]), file=sys.stderr, flush=True)
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"color_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
