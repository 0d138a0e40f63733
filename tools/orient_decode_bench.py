#!/usr/bin/env python
"""Oriented decode against decode and decode + xpngb_transform on the GPU; one JSON line to profiles/orient_decode_<tag>.json.

  A  the bench.py workload (1000 sintel-like 1080p frames, seeds 1000..1999), levels 1 and 2, R90 for every entry: ms per
     call of xpngb_decode, xpngb_decode_oriented, and xpngb_decode followed by xpngb_transform, with files and pixels in
     device memory and again in pinned host memory.
  B  the same frames, one seeded 224 x 224 crop each, ops drawn from {MH, TL}: xpngb_decode_region against
     xpngb_decode_oriented (device memory).
  C  rgb_4k_s1 and rgba_8192_s2, full image, R90, the three paths of A (device and host memory).

Before anything is timed, every oriented output is compared with decode (or decode_region) + xpngb_transform of the same
files.  A timing is 3 warm-up calls and then `--reps` calls, each ending in a device synchronise; median and minimum are
reported, with xpngb_last_kernel_ms of the last call (for decode + transform: the sum of both calls).
Usage: python tools/orient_decode_bench.py [--frames 1000] [--reps 7] [--tag b200]"""
import argparse
import ctypes as C
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
from xpng_b200.codec import OPS, _Image, lib, op_codes, rects  # noqa: E402
from conftest import make_case, manifest  # noqa: E402


def copy_descs(d):
    """A fresh copy of a descriptor array (xpngb_transform swaps w and h of the quarter turns in place)."""
    t = (_Image * len(d))()
    C.memmove(t, d, C.sizeof(d))
    return t


def buffers(nbytes, dev):
    mk = (lambda: torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda")) if dev else \
        (lambda: torch.zeros(nbytes + 64, dtype=torch.uint8).pin_memory())
    return mk(), mk()


def transform(cd, op, descs, n, src, size, dst, dev):
    if lib().xpngb_transform(cd._h, OPS[op], copy_descs(descs), n, C.c_void_p(src), size, int(dev), C.c_void_p(dst), int(dev)):
        raise RuntimeError("xpngb_transform: " + cd._err())
    return cd.last_kernel_ms


def three_paths(cd, B, op, dev, reps):
    """Whole images, the same op for every entry: decode, decode_oriented, decode + transform."""
    d, total = B.descs()
    fptr = B.dev.data_ptr() if dev else B.host.ctypes.data
    plain, turned = buffers(total, dev)
    ops = op_codes([op] * B.n)
    ms = {}

    def dec():
        cd.decode_raw(d, B.n, fptr, B.fsize, int(dev), B.foffs, B.fsizes, plain.data_ptr(), total, int(dev))
        ms["dec"] = cd.last_kernel_ms

    def ori():
        cd.decode_oriented_raw(d, ops, None, B.n, fptr, B.fsize, int(dev), B.foffs, B.fsizes, turned.data_ptr(), total, int(dev))

    def dec_tr():
        dec()
        ms["tr"] = transform(cd, op, d, B.n, plain.data_ptr(), total, ref.data_ptr(), dev)

    ref = turned.clone() if dev else torch.zeros_like(turned).pin_memory()
    ori(); dec_tr(); torch.cuda.synchronize()
    if not torch.equal(turned, ref):
        raise SystemExit(f"parity: oriented decode ({op}) differs from decode + xpngb_transform")
    out = {}
    out["decode"] = timed(dec, reps); out["decode"]["kernel_ms"] = round(ms["dec"], 3)
    out["decode_oriented"] = timed(ori, reps); out["decode_oriented"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["decode_then_transform"] = timed(dec_tr, reps)
    out["decode_then_transform"]["kernel_ms"] = round(ms["dec"] + ms["tr"], 3)
    out["transform_kernel_ms"] = round(ms["tr"], 3)
    for k in ("decode_oriented", "decode_then_transform"):
        out[k]["over_decode_ms"] = round(out[k]["median_ms"] - out["decode"]["median_ms"], 3)
    out["pixels_bytes"] = total
    return out


def crops_mixed_ops(cd, B, boxes, ops, reps):
    """B: decode_region against decode_oriented with per-entry ops (device memory)."""
    d, total = B.descs(boxes)
    ra, oa = rects(boxes), op_codes(ops)
    region, turned = buffers(total, True)
    fptr = B.dev.data_ptr()

    def reg():
        cd.decode_region_raw(d, ra, B.n, fptr, B.fsize, 1, B.foffs, B.fsizes, region.data_ptr(), total, 1)

    def ori():
        cd.decode_oriented_raw(d, oa, ra, B.n, fptr, B.fsize, 1, B.foffs, B.fsizes, turned.data_ptr(), total, 1)

    reg(); ori(); torch.cuda.synchronize()
    ref = region.clone()                      # decode_region + xpngb_transform of the entries that are not copies
    for op in set(ops) - {"tl", "tr"}:
        idx = [i for i, o in enumerate(ops) if o == op]
        sub = (_Image * len(idx))()
        for k, i in enumerate(idx):
            sub[k].w, sub[k].h, sub[k].A, sub[k].offset = boxes[i][2], boxes[i][3], d[i].A, d[i].offset
        transform(cd, op, sub, len(idx), region.data_ptr(), total, ref.data_ptr(), True)
    torch.cuda.synchronize()
    if not torch.equal(turned, ref):
        raise SystemExit("parity: oriented region decode differs from decode_region + xpngb_transform")
    out = {"decode_region": timed(reg, reps)}
    out["decode_region"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["decode_oriented"] = timed(ori, reps)
    out["decode_oriented"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["time_ratio"] = round(out["decode_oriented"]["median_ms"] / out["decode_region"]["median_ms"], 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("orient_decode_bench needs a CUDA device")
    res = {"tool": "tools/orient_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3}
    cd = xpng_b200.Codec(0)

    # ---- A and B: the bench.py batch
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    rng = np.random.default_rng(2027)
    boxes = [(int(rng.integers(1920 - 224 + 1)), int(rng.integers(1080 - 224 + 1)), 224, 224) for _ in frames]
    ops = [("mh", "tl")[int(rng.integers(2))] for _ in frames]
    files = {}
    for lv in (1, 2):
        files[lv] = []
        for k in range(0, len(frames), 250):
            files[lv] += cd.encode(lv, frames[k: k + 250])
    del frames
    A, Bres = {"frames": a.frames, "op": "r90"}, {"frames": a.frames, "crop": [224, 224], "ops": "mh or tl, seeded",
                                                  "mh_entries": ops.count("mh")}
    for lv in (1, 2):
        B = Batch(files[lv])
        for where, dev in (("device", True), ("host", False)):
            A[f"L{lv}_{where}"] = three_paths(cd, B, "r90", dev, a.reps)
            print(json.dumps({"A": {f"L{lv}_{where}": A[f"L{lv}_{where}"]}}), file=sys.stderr, flush=True)
        Bres[f"L{lv}"] = crops_mixed_ops(cd, B, boxes, ops, a.reps)
        print(json.dumps({"B": {f"L{lv}": Bres[f"L{lv}"]}}), file=sys.stderr, flush=True)
        del B
    res["A_batch_r90"] = A
    res["B_crops_mh_tl"] = Bres
    del files

    # ---- C: single large images
    man = manifest()["synthetic"]
    Cres = {}
    for name in ("rgb_4k_s1", "rgba_8192_s2"):
        px = make_case("synthetic", name, man[name])
        for lv in (1, 2):
            B = Batch(cd.encode(lv, [px]))
            for where, dev in (("device", True), ("host", False)):
                Cres[f"{name}_L{lv}_{where}"] = three_paths(cd, B, "r90", dev, a.reps)
                print(json.dumps({"C": {f"{name}_L{lv}_{where}": Cres[f"{name}_L{lv}_{where}"]}}), file=sys.stderr, flush=True)
            del B
    res["C_single_r90"] = Cres
    cd.close()
    out = os.path.join(ROOT, "profiles", f"orient_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
