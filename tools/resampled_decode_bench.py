#!/usr/bin/env python
"""Resampled decode on the GPU; one JSON line to profiles/resampled_decode_<tag>.json.  Files and outputs in device memory.

  a  no regression: 1000 sintel-like 1080p frames, one seeded RandomResizedCrop box each, bilinear to 224 x 224 at level
     1, through xpngb_decode_resized and through xpngb_decode_resampled with filters == NULL (same bytes, checked)
  b  the same boxes resized to 224 x 224 with every filter, at levels 1 and 2
  c  the eval transform Resize(256) + CenterCrop(224) to a normalised float32 (N, 3, 224, 224) tensor: one
     xpngb_decode_resampled call with windows (bilinear and bicubic), against today's best path, a ragged
     decode_tensor_raw of the whole 256-short images (bilinear only) followed by a torch slice and stack
The arms of a and of c alternate call by call.  A sample of every path is compared with tests/test_resampled_decode.py's
resize_pil first.  Each timing is 3 warm-up calls, then --reps calls per arm, each ending in a device synchronise.
Usage: python tools/resampled_decode_bench.py [--frames 1000] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, filter_codes, rects, resize_center_crop, sizes, tensor_format  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import rrc_boxes  # noqa: E402
from test_resampled_decode import FILTERS, resize_pil, window  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from resized_decode_bench import buf, out_descs  # noqa: E402

OUT = (224, 224)
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
NAMES = {1: "lanczos", 2: "bilinear", 3: "bicubic", 4: "box", 5: "hamming"}


def alternate(fns, reps):
    """{name: median / min ms}, the arms called in turn, each call ending in a device synchronise."""
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return {k: {"median_ms": round(float(np.median(v)), 3), "min_ms": round(float(np.min(v)), 3)} for k, v in ts.items()}


def sample(files, boxes, f, wins, got, k=250):
    for i in range(0, len(files), k):
        full = po.decode(files[i])
        x, y, w, h = boxes[i] if boxes is not None else (0, 0, full.shape[1], full.shape[0])
        yield i, full[y: y + h, x: x + w], got(i)


def arm_a_b(cd, B, files, boxes, reps, lv):
    n = B.n
    ra, sa = rects(boxes), sizes([OUT] * n)
    d, tot = out_descs(B, [OUT] * n)
    u_old, u_new = buf(tot, True), buf(tot, True)
    fptr = B.dev.data_ptr()
    old = lambda: cd.decode_resized_raw(d, None, ra, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u_old.data_ptr(), tot, 1)
    res = {}
    if lv == 1:
        new = lambda: cd.decode_resampled_raw(None, d, None, None, ra, sa, None, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u_new.data_ptr(), tot, 1)
        old(); new(); torch.cuda.synchronize()
        if not torch.equal(u_old, u_new):
            raise SystemExit("a: xpngb_decode_resampled(filters=NULL) differs from xpngb_decode_resized")
        res["a_bilinear_L1"] = alternate({"decode_resized": old, "decode_resampled_null_filters": new}, reps)
    b = {}
    for f in FILTERS:
        fa = filter_codes(f, n)
        call = lambda: cd.decode_resampled_raw(None, d, fa, None, ra, sa, None, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u_new.data_ptr(), tot, 1)
        call(); torch.cuda.synchronize()
        host = u_new.cpu().numpy()
        for i, crop, g in sample(files, boxes, f, None, lambda i: host[d[i].offset: d[i].offset + OUT[0] * OUT[1] * 3].reshape(OUT[1], OUT[0], 3)):
            if not np.array_equal(g, resize_pil(crop, *OUT, f)):
                raise SystemExit(f"b: {NAMES[f]} entry {i} differs from resize_pil")
        b[NAMES[f]] = alternate({"decode_resampled": call}, reps)["decode_resampled"]
        b[NAMES[f]]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    res[f"b_rrc_224_L{lv}"] = b
    return res


def arm_c(cd, B, files, reps):
    n = B.n
    geo = [resize_center_crop(w, h, 256, 224) for (w, h, _) in B.hdr]
    szs, wins = [z for z, _ in geo], [w for _, w in geo]
    fmt = tensor_format("float32", "chw", "div", MEAN, STD)
    per = 3 * 224 * 224
    t = torch.empty((n, 3, 224, 224), dtype=torch.float32, device="cuda")
    td = (_Image * n)()
    for i in range(n):
        td[i].offset = i * per * 4
    # today: ragged tensors of the whole resized images, then a slice and a stack
    rd, off = (_Image * n)(), 0
    for i, (W, H) in enumerate(szs):
        rd[i].offset = off
        off += (3 * W * H * 4 + 15) & ~15
    rag = torch.empty(off // 4 + 16, dtype=torch.float32, device="cuda")
    views = [rag[rd[i].offset // 4: rd[i].offset // 4 + 3 * W * H].view(3, H, W)[:, y: y + ch, x: x + cw]
             for i, ((W, H), (x, y, cw, ch)) in enumerate(zip(szs, wins))]
    sa, wa, fptr = sizes(szs), rects(wins), B.dev.data_ptr()

    def today():
        cd.decode_tensor_raw(fmt, rd, None, None, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, rag.data_ptr(), off, 1)
        return torch.stack(views)

    def one_call(f):
        fa = filter_codes(f, n)
        return lambda: cd.decode_resampled_raw(fmt, td, fa, None, None, sa, wa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t.data_ptr(), n * per * 4, 1)

    for f in (2, 3):
        one_call(f)(); torch.cuda.synchronize()
        for i, px, g in sample(files, None, f, wins, lambda i: t[i]):
            want = to_tensor_ref(window(resize_pil(px, *szs[i], f), wins[i]), "float32", "chw", "div", MEAN, STD)
            if not np.array_equal(bits(g), want):
                raise SystemExit(f"c: {NAMES[f]} entry {i} differs from the reference")
    one_call(2)(); ref = today(); torch.cuda.synchronize()
    if not torch.equal(ref.view(torch.int32), t.view(torch.int32)):
        raise SystemExit("c: the one-call bilinear tensor differs from today's path")
    r = alternate({"today_ragged_tensor_slice_stack_bilinear": today, "decode_resampled_window_bilinear": one_call(2),
                   "decode_resampled_window_bicubic": one_call(3)}, reps)
    return {"resized": sorted(set(szs)), "window": sorted(set(w[2:] for w in wins)), **r}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/resampled_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("resampled_decode_bench needs a CUDA device")
    res = {"tool": "tools/resampled_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "frames": a.frames, "size": list(OUT)}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    boxes = rrc_boxes(np.random.default_rng(2029), len(frames))
    for lv in (1, 2):
        files = []
        for k in range(0, len(frames), 250):
            files += cd.encode(lv, frames[k: k + 250])
        B = Batch(files)
        res.update(arm_a_b(cd, B, files, boxes, a.reps, lv))
        if lv == 1:
            res["c_eval_resize256_crop224_f32_L1"] = arm_c(cd, B, files, a.reps)
        print(json.dumps({k: v for k, v in res.items() if k.endswith(f"L{lv}")}), file=sys.stderr, flush=True)
        del B
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"resampled_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
