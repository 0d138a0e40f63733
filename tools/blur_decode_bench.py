#!/usr/bin/env python
"""Blurred and solarized decode on the GPU; one JSON line to profiles/blur_decode_<tag>.json.  Files and outputs in device memory.

The workload is the colour bench's BYOL batch (sintel-like 1080p frames at levels 1 and 2, a seeded RandomResizedCrop box
resized to 224 x 224, flip p 0.5, ColorJitter(0.4, 0.4, 0.2, 0.1) p 0.8, RandomGrayscale p 0.2, ImageNet-normalised float32
(N, 3, 224, 224)), followed by BYOL's second view: GaussianBlur (radius uniform in [0.1, 2.0]) with p 0.1 and solarize with p
0.2; a second variant blurs every entry (p 1.0).  The arms, called in turn:
  color   the colour transform without blur and solarize, one xpngb_decode_color call: the floor
  blur    the whole view in one xpngb_decode_blur call
  pil     uint8 colour decode (xpngb_decode_color), the pixels to the host, PIL's GaussianBlur and solarize per entry, back to
          the device, then ToTensor + Normalize there
A sample of the blur arm is compared with Pillow first.  Each timing is 3 warm-up calls, then --reps calls per arm, each ending
in a device synchronise; the median is reported.  Per-kernel times of one blur call come from xpngb_profile.
Usage: python tools/blur_decode_bench.py [--frames 1000] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
from PIL import Image, ImageFilter, ImageOps  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, blur_array, blur_params, color_array, op_codes, rects, sizes, tensor_format  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import rrc_boxes  # noqa: E402
from test_resampled_decode import resize_pil  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from test_color_decode import color_ref  # noqa: E402
from resampled_decode_bench import alternate  # noqa: E402
from color_decode_bench import programs  # noqa: E402

OUT = (224, 224)
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def blur_programs(n, seed, blur_p, sol_p=0.2):
    """Blur entry per frame, drawn as BYOL's RandomApply([GaussianBlur], p) and RandomSolarize(p) draw them."""
    rng = random.Random(seed)
    out = []
    for _ in range(n):
        radius = rng.uniform(0.1, 2.0) if rng.random() < blur_p else None
        thr = 128 if rng.random() < sol_p else None
        out.append(None if radius is None and thr is None else blur_params(radius, thr))
    return out


def pil_blur(px, b):
    if b is None:
        return px
    im = Image.fromarray(px)
    if b.radius[0]:
        im = im.filter(ImageFilter.GaussianBlur(b.radius[0]))
    if b.solarize:
        im = ImageOps.solarize(im, b.threshold)
    return np.asarray(im)


def run_level(cd, files, boxes, ops, cols, blurs, reps):
    n = len(files)
    B = Batch(files)
    fptr = B.dev.data_ptr()
    ra, sa, oa, ca, ba = rects(boxes), sizes([OUT] * n), op_codes(ops), color_array(cols, n), blur_array(blurs, n)
    fmt = tensor_format("float32", "chw", "div", MEAN, STD, drop_alpha=True)
    per = 3 * OUT[0] * OUT[1]
    td = (_Image * n)()
    ud = (_Image * n)()
    for i in range(n):
        td[i].offset = i * per * 4
        ud[i].offset = i * per
    t_col = torch.empty((n, 3, *OUT[::-1]), dtype=torch.float32, device="cuda")
    t_blur = torch.empty_like(t_col)
    u8 = torch.empty((n, OUT[1], OUT[0], 3), dtype=torch.uint8, device="cuda")
    host = torch.empty((n, OUT[1], OUT[0], 3), dtype=torch.uint8).pin_memory()
    mean = torch.tensor(MEAN, device="cuda").view(3, 1, 1)
    std = torch.tensor(STD, device="cuda").view(3, 1, 1)

    color = lambda: cd.decode_color_raw(fmt, td, None, oa, ra, sa, None, ca, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t_col.data_ptr(), n * per * 4, 1)
    blur = lambda: cd.decode_blur_raw(fmt, td, None, oa, ra, sa, None, ca, ba, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t_blur.data_ptr(),
                                      n * per * 4, 1)

    def pil():
        cd.decode_color_raw(None, ud, None, oa, ra, sa, None, ca, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u8.data_ptr(), n * per, 1)
        host.copy_(u8)
        h = host.numpy()
        for i in range(n):
            if blurs[i] is not None:
                h[i] = pil_blur(h[i], blurs[i])
        return host.cuda(non_blocking=True).permute(0, 3, 1, 2).float().div_(255).sub_(mean).div_(std)

    blur(); torch.cuda.synchronize()
    for i in range(0, n, max(1, n // 40)):   # the blur arm against Pillow on a sample
        x, y, w, h = boxes[i]
        px = po.orient(ops[i], resize_pil(po.decode(files[i])[y: y + h, x: x + w], *OUT, 2))
        want = pil_blur(px if cols[i] is None else color_ref(px, cols[i]), blurs[i])
        if not np.array_equal(bits(t_blur[i]), to_tensor_ref(want, "float32", "chw", "div", MEAN, STD)):
            raise SystemExit(f"entry {i}: blur decode differs from Pillow")
    cd.profile(True)
    blur()
    prof = {k: v for k, v in cd.profile_report().items() if k.startswith(("k_color", "k_blur", "k_to_tensor"))}
    cd.profile(False)
    r = alternate({"color": color, "blur": blur, "pil": pil}, reps)
    r["blur_adds_ms"] = round(r["blur"]["median_ms"] - r["color"]["median_ms"], 3)
    r["profiled_one_blur_call_ms"] = {k: [round(v[0], 3), v[1]] for k, v in prof.items()}
    r["blurred_entries"] = sum(b is not None and b.radius[0] > 0 for b in blurs)
    r["solarized_entries"] = sum(b is not None and b.solarize for b in blurs)
    del B
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/blur_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 7:
        raise SystemExit("--reps must be at least 7")
    if not torch.cuda.is_available():
        raise SystemExit("blur_decode_bench needs a CUDA device")
    res = {"tool": "tools/blur_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "frames": a.frames, "size": list(OUT)}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    boxes = rrc_boxes(np.random.default_rng(2029), len(frames))
    ops, cols = programs(len(frames), 2030)
    for lv in (1, 2):
        files = []
        for k in range(0, len(frames), 250):
            files += cd.encode(lv, frames[k: k + 250])
        for name, p in (("byol_view2", 0.1), ("blur_all", 1.0)):
            key = f"{name}_224_f32_L{lv}"
            res[key] = run_level(cd, files, boxes, ops, cols, blur_programs(len(frames), 2031, p), a.reps)
            print(json.dumps(res[key]), file=sys.stderr, flush=True)
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"blur_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
