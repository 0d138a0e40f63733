#!/usr/bin/env python
"""Multi-view decode on the GPU; one JSON line to profiles/views_decode_<tag>.json.  Files and outputs in device memory.

Workloads (every view ImageNet-normalised float32 (N, 3, s, s), bicubic RandomResizedCrop, flip p 0.5, ColorJitter(0.4, 0.4,
0.2, 0.1) p 0.8, RandomGrayscale p 0.2, GaussianBlur with DINO's per-view probabilities; draws from seeded torch and Python
RNGs as DINO draws them):
  A  dino_1080p   DINO 2 x 224 (scale 0.4-1) + 10 x 96 (scale 0.05-0.4) on bench.py's sintel-like 1080p frames
  B  byol_1080p   BYOL's two views, 2 x 224 (scale 0.08-1), on the same frames
  C  dino_500x375 DINO 2 + 10 on seeded 500 x 375 images (one tile each)
each at levels 1 and 2.  The arms, called in turn:
  per_view     one xpngb_decode_blur call per view (the recipe without multi-view decode): every view decodes its own tiles
  own_offsets  one call with every view's entries, each view reading its own copy of the files (no entries share a file)
  shared       one call with every view's entries reading the same files: what Codec.decode_views issues
All three arms' outputs are compared byte for byte, and a sample of the shared arm with Pillow, before any timing.  Each
timing is 3 warm-up calls, then --reps calls per arm, each ending in a device synchronise; the median is reported, with the
arm's xpngb_last_tiles (summed over its calls), which must equal the tile counts recomputed here from the draws.
Usage: python tools/views_decode_bench.py [--frames 1000] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import torchvision.transforms as T  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, blur_array, color_array, filter_codes, op_codes, rects, region_tiles, sizes, tensor_format  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resampled_decode import resize_pil  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from test_color_decode import color_ref  # noqa: E402
from test_blur_decode import _replay_view, pil_blur  # noqa: E402
from resampled_decode_bench import alternate  # noqa: E402

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
BICUBIC = 3
DINO = [(224, (0.4, 1.0), 1.0, 0.0), (224, (0.4, 1.0), 0.1, 0.2)] + [(96, (0.05, 0.4), 0.5, 0.0)] * 10   # size, scale, blur p, solarize p
BYOL = [(224, (0.08, 1.0), 1.0, 0.0), (224, (0.08, 1.0), 0.1, 0.2)]


def draws(views, whs, seed):
    """Per view, per image: (box, op, colour, blur) replayed from torch's and Python's RNGs."""
    torch.manual_seed(seed)
    random.seed(seed)
    cj = T.ColorJitter(0.4, 0.4, 0.2, 0.1)
    out = [[] for _ in views]
    for w, h in whs:
        stand_in = torch.zeros(1, 1, 1).expand(3, h, w)   # get_params reads the size only
        for v, (s, scale, bp, sp) in enumerate(views):
            out[v].append(_replay_view(T.RandomResizedCrop(s, scale=scale), stand_in, cj, bp, sp))
    return out


def tile_counts(whs, dr):
    per_view = sum(region_tiles(w, h, d[k][0])[0] for d in dr for k, (w, h) in enumerate(whs))
    once = 0
    for k, (w, h) in enumerate(whs):
        bx = [d[k][0] for d in dr]
        x0, y0 = min(b[0] for b in bx), min(b[1] for b in bx)
        once += region_tiles(w, h, (x0, y0, max(b[0] + b[2] for b in bx) - x0, max(b[1] + b[3] for b in bx) - y0))[0]
    return per_view, once


def run(cd, files, whs, views, dr, reps):
    n, nv = len(files), len(views)
    B = Batch(files)
    fmt = tensor_format("float32", "chw", "div", MEAN, STD, drop_alpha=True)
    outs = [torch.empty((n, 3, s, s), dtype=torch.float32, device="cuda") for s, _, _, _ in views]
    outs_all = [torch.empty_like(o) for o in outs]
    # one call per view
    per_view = []
    for v, (s, _, _, _) in enumerate(views):
        d = dr[v]
        td = (_Image * n)()
        for i in range(n):
            td[i].offset = i * 3 * s * s * 4
        a = (td, filter_codes(BICUBIC, n), op_codes([x[1] for x in d]), rects([x[0] for x in d]), sizes([(s, s)] * n), None,
             color_array([x[2] for x in d], n), blur_array([x[3] for x in d], n))
        per_view.append((a, outs[v]))

    def call_per_view():
        t = 0
        for a, o in per_view:
            cd.decode_blur_raw(fmt, *a, n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, o.data_ptr(), o.numel() * 4, 1)
            t += cd.last_tiles
        return t

    # every view in one call: entry v * n + i is view v of file i, written into its view's tensor
    m = n * nv
    flat = [torch.empty(sum(o.numel() for o in outs), dtype=torch.float32, device="cuda") for _ in range(2)]
    td = (_Image * m)()
    at = 0
    for v, (s, _, _, _) in enumerate(views):
        for i in range(n):
            td[v * n + i].offset = (at + i * 3 * s * s) * 4
        at += n * 3 * s * s
    allv = [x for d in dr for x in d]
    a = (td, filter_codes(BICUBIC, m), op_codes([x[1] for x in allv]), rects([x[0] for x in allv]),
         sizes([(s, s) for s, _, _, _ in views for _ in range(n)]), None, color_array([x[2] for x in allv], m),
         blur_array([x[3] for x in allv], m))
    shared_offs, shared_sizes = (C.c_uint64 * m)(), (C.c_uint64 * m)()
    own_offs = (C.c_uint64 * m)()
    copies = torch.empty(nv * B.fsize + 64, dtype=torch.uint8, device="cuda")   # view v reads copy v of the files
    for v in range(nv):
        copies[v * B.fsize: (v + 1) * B.fsize].copy_(B.dev[: B.fsize])
        for i in range(n):
            shared_offs[v * n + i], shared_sizes[v * n + i] = B.foffs[i], B.fsizes[i]
            own_offs[v * n + i] = v * B.fsize + B.foffs[i]
    torch.cuda.synchronize()

    def call_shared():
        cd.decode_blur_raw(fmt, *a, m, B.dev.data_ptr(), B.fsize, 1, shared_offs, shared_sizes, flat[0].data_ptr(), flat[0].numel() * 4, 1)
        return cd.last_tiles

    def call_own():
        cd.decode_blur_raw(fmt, *a, m, copies.data_ptr(), nv * B.fsize, 1, own_offs, shared_sizes, flat[1].data_ptr(), flat[1].numel() * 4, 1)
        return cd.last_tiles

    tiles = {"per_view": call_per_view(), "own_offsets": call_own(), "shared": call_shared()}
    torch.cuda.synchronize()
    want_per_view, want_once = tile_counts(whs, dr)
    if tiles != {"per_view": want_per_view, "own_offsets": want_per_view, "shared": want_once}:
        raise SystemExit(f"tile counts {tiles} differ from the draws' {want_per_view} per view, {want_once} once per file")
    at = 0
    for v, o in enumerate(outs):   # parity: the three arms byte for byte, then a sample of the shared arm against Pillow
        k = o.numel()
        if not (torch.equal(flat[0][at: at + k].view(torch.int32), o.view(-1).view(torch.int32))
                and torch.equal(flat[1][at: at + k].view(torch.int32), o.view(-1).view(torch.int32))):
            raise SystemExit(f"view {v}: the arms' outputs differ")
        outs_all[v].view(-1).copy_(flat[0][at: at + k])
        at += k
    for v in (0, 1, nv - 1):
        s = views[v][0]
        for i in range(0, n, max(1, n // 4)):
            box, op, c, b = dr[v][i]
            x, y, w, h = box
            px = po.orient(op, resize_pil(po.decode(files[i])[y: y + h, x: x + w], s, s, BICUBIC))
            px = pil_blur(px if c is None else color_ref(px, c), b)
            if not np.array_equal(bits(outs_all[v][i]), to_tensor_ref(px, "float32", "chw", "div", MEAN, STD)):
                raise SystemExit(f"view {v} entry {i}: shared decode differs from Pillow")
    r = alternate({"per_view": call_per_view, "own_offsets": call_own, "shared": call_shared}, reps)
    for k in r:
        r[k]["tiles"] = tiles[k]
    r["entries"] = m
    r["shared_vs_per_view"] = round(r["per_view"]["median_ms"] / r["shared"]["median_ms"], 3)
    r["shared_vs_own_offsets"] = round(r["own_offsets"]["median_ms"] / r["shared"]["median_ms"], 3)
    del B, copies, flat
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/views_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 7:
        raise SystemExit("--reps must be at least 7")
    if not torch.cuda.is_available():
        raise SystemExit("views_decode_bench needs a CUDA device")
    res = {"tool": "tools/views_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "frames": a.frames}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))   # bench.py's frames (SEED0 = 1000)
    small = [synth.rgb(375, 500, 5000 + k) for k in range(a.frames)]
    for name, imgs, views, seed in (("dino_1080p", frames, DINO, 2040), ("byol_1080p", frames, BYOL, 2041),
                                    ("dino_500x375", small, DINO, 2042)):
        whs = [(im.shape[1], im.shape[0]) for im in imgs]
        dr = draws(views, whs, seed)
        for lv in (1, 2):
            files = []
            for k in range(0, len(imgs), 250):
                files += cd.encode(lv, imgs[k: k + 250])
            key = f"{name}_L{lv}"
            res[key] = run(cd, files, whs, views, dr, a.reps)
            print(key, json.dumps(res[key]), file=sys.stderr, flush=True)
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"views_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
