#!/usr/bin/env python
"""Tensor decode against the torch conversion callers write today, on the GPU; one JSON line to profiles/tensor_decode_<tag>.json.

  A  the bench.py workload (1000 sintel-like 1080p frames, seeds 1000..), levels 1 and 2, files and output in device memory,
     one seeded RandomResizedCrop-style box per frame resized to 224 x 224, MH on a seeded half (TL on the rest):
       today_f32 / today_f16   xpngb_decode_resized, then per-entry views, stack, permute, float, div(255), normalize with
                               ImageNet mean / std (and .half() for f16): what a training loader does with the uint8 output
       tensor_f32 / tensor_f16 xpngb_decode_tensor, (N, 3, 224, 224) CHW, scale "div", the same normalisation
  B  whole 1080p frames (the first --frames-b of A's), no resize, F16 CHW: xpngb_decode + the torch conversion against
     xpngb_decode_tensor.  Every tensor entry takes a pass through a decode window that the plain decode writes in place.
  K  k_to_tensor's own time (xpngb_profile: launches serialised, a run of its own) for A at level 1, f32 and f16, and the
     bytes it must move (uint8 source in, tensor out, from the shapes) over that time, against 7.7 TB/s.

Before anything is timed, a sample of every path's outputs is compared bit for bit with tests/test_tensor_decode.py's
to_tensor_ref.  A timing is 3 warm-up calls and then `--reps` calls, each ending in a device synchronise; median and
minimum are reported, with xpngb_last_kernel_ms of the last call for the library paths.
Usage: python tools/tensor_decode_bench.py [--frames 1000] [--frames-b 200] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info, timed  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, op_codes, rects, sizes, tensor_format  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import resize_bilinear, rrc_boxes  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from resized_decode_bench import buf, out_descs  # noqa: E402

OUT = (224, 224)
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
HBM_TBPS = 7.7


def tensor_descs(n, per_bytes):
    arr = (_Image * n)()
    for i in range(n):
        arr[i].offset = i * per_bytes
    return arr


def torch_convert(views, half):
    """The conversion a loader writes after a uint8 HWC decode: stack, permute, float, div(255), normalize, cast."""
    x = torch.stack(views).permute(0, 3, 1, 2).float().div(255)
    m = torch.tensor(MEAN, device=x.device).view(1, 3, 1, 1)
    s = torch.tensor(STD, device=x.device).view(1, 3, 1, 1)
    x = x.sub(m).div(s)
    return x.half() if half else x


def check_sample(files, boxes, ops, got, dt, k):
    for i in range(0, len(files), k):
        full = po.decode(files[i])
        x, y, w, h = boxes[i] if boxes is not None else (0, 0, full.shape[1], full.shape[0])
        px = full[y: y + h, x: x + w]
        if boxes is not None:
            px = resize_bilinear(px, *OUT)
        want = to_tensor_ref(po.orient(ops[i] if ops else "tl", px), dt, "chw", "div", MEAN, STD)
        if not np.array_equal(bits(got[i]), want):
            raise SystemExit(f"parity: {dt} entry {i} differs from to_tensor_ref")


def batch_a(cd, B, files, boxes, ops, reps):
    n = B.n
    ra, oa, sa = rects(boxes), op_codes(ops), sizes([OUT] * n)
    fptr = B.dev.data_ptr()
    dr, tr = out_descs(B, [OUT] * n)
    u8 = buf(tr, True)
    views = [u8[d.offset: d.offset + OUT[0] * OUT[1] * 3].view(OUT[1], OUT[0], 3) for d in dr]
    out = {}
    for dt, half in (("float32", False), ("float16", True)):
        eb = 2 if half else 4
        per = 3 * OUT[0] * OUT[1]
        t = torch.empty((n, 3, OUT[1], OUT[0]), dtype=getattr(torch, dt), device="cuda")
        td, fmt = tensor_descs(n, per * eb), tensor_format(dt, "chw", "div", MEAN, STD)

        def today():
            cd.decode_resized_raw(dr, oa, ra, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u8.data_ptr(), tr, 1)
            return torch_convert(views, half)

        def tensor():
            cd.decode_tensor_raw(fmt, td, oa, ra, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t.data_ptr(), n * per * eb, 1)

        tensor(); torch.cuda.synchronize()
        check_sample(files, boxes, ops, t, dt, 50)
        ref = today(); torch.cuda.synchronize()
        # the torch conversion is not the contract (its division by std is the GPU's own); report how far it is from it
        out[f"today_vs_tensor_{dt}_differing_elements"] = int((bits(ref) != bits(t)).sum())
        out[f"today_{dt}"] = timed(today, reps)
        out[f"today_{dt}"]["decode_kernel_ms"] = round(cd.last_kernel_ms, 3)
        out[f"tensor_{dt}"] = timed(tensor, reps)
        out[f"tensor_{dt}"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
        del t
    return out


def batch_b(cd, B, files, reps):
    n = B.n
    fptr = B.dev.data_ptr()
    df, tf = B.descs()
    u8 = buf(tf, True)
    views = [u8[d.offset: d.offset + w * h * c].view(h, w, c) for d, (w, h, c) in zip(df, B.hdr)]
    W, H, _ = B.hdr[0]
    per = 3 * W * H
    t = torch.empty((n, 3, H, W), dtype=torch.float16, device="cuda")
    td, fmt = tensor_descs(n, per * 2), tensor_format("float16", "chw", "div", MEAN, STD)

    def today():
        cd.decode_raw(df, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u8.data_ptr(), tf, 1)
        return torch_convert(views, True)

    def tensor():
        cd.decode_tensor_raw(fmt, td, None, None, None, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t.data_ptr(), n * per * 2, 1)

    tensor(); torch.cuda.synchronize()
    check_sample(files, None, None, t, "float16", 25)
    out = {"frames": n, "today_decode_plus_torch_f16": timed(today, reps)}
    out["today_decode_plus_torch_f16"]["decode_kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["tensor_f16"] = timed(tensor, reps)
    out["tensor_f16"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    return out


def kernel_rate(cd, B, boxes, ops):
    n = B.n
    ra, oa, sa = rects(boxes), op_codes(ops), sizes([OUT] * n)
    res = {}
    for dt, eb in (("float32", 4), ("float16", 2)):
        per = 3 * OUT[0] * OUT[1]
        t = torch.empty(n * per * eb, dtype=torch.uint8, device="cuda")
        td, fmt = tensor_descs(n, per * eb), tensor_format(dt, "chw", "div", MEAN, STD)
        cd.profile(True)
        calls = 3
        for _ in range(calls):
            cd.decode_tensor_raw(fmt, td, oa, ra, sa, n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, t.data_ptr(), n * per * eb, 1)
        rep = cd.profile_report()
        cd.profile(False)
        ms, cnt = rep.get("k_to_tensor", (0.0, 0))
        per_call = ms / calls
        nbytes = n * per * (1 + eb)                 # the resized uint8 pixels in, the tensor out
        res[dt] = {"k_to_tensor_ms_per_call": round(per_call, 4), "launches_per_call": cnt // calls, "bytes": nbytes,
                   "GB_per_s": round(nbytes / per_call / 1e6, 1) if per_call else None,
                   "share_of_7.7_TBps": round(nbytes / per_call / 1e9 / HBM_TBPS, 3) if per_call else None,
                   "all_kernels_ms_per_call": round(sum(v[0] for v in rep.values()) / calls, 3)}
        del t
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--frames-b", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/tensor_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("tensor_decode_bench needs a CUDA device")
    res = {"tool": "tools/tensor_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "size": list(OUT),
           "mean": MEAN, "std": STD}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    rng = np.random.default_rng(2028)
    boxes = rrc_boxes(rng, len(frames))
    ops = [("mh", "tl")[int(rng.integers(2))] for _ in frames]
    files = {}
    for lv in (1, 2):
        files[lv] = []
        for k in range(0, len(frames), 250):
            files[lv] += cd.encode(lv, frames[k: k + 250])
    del frames
    A = {"frames": a.frames, "boxes": "RandomResizedCrop-style, seeded", "mh_entries": ops.count("mh")}
    for lv in (1, 2):
        B = Batch(files[lv])
        A[f"L{lv}_device"] = batch_a(cd, B, files[lv], boxes, ops, a.reps)
        print(json.dumps({"A": {f"L{lv}_device": A[f"L{lv}_device"]}}), file=sys.stderr, flush=True)
        if lv == 1:
            res["K_to_tensor_L1_device"] = kernel_rate(cd, B, boxes, ops)
            print(json.dumps({"K": res["K_to_tensor_L1_device"]}), file=sys.stderr, flush=True)
        del B
    res["A_batch_rrc_224"] = A
    Bres = {}
    for lv in (1, 2):
        fb = files[lv][: a.frames_b]
        B = Batch(fb)
        Bres[f"L{lv}_device"] = batch_b(cd, B, fb, a.reps)
        print(json.dumps({"B": {f"L{lv}_device": Bres[f"L{lv}_device"]}}), file=sys.stderr, flush=True)
        del B
    res["B_whole_1080p_f16"] = Bres
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"tensor_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
